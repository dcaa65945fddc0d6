"""Kernels at the largest sizes their entry points accept (just under 2^31 elements), and the drop-in classes just over.

The kernels index in 32 bits behind a host check of < 2^31 elements, so a grid-stride loop whose count lies within one
stride of 2^31 must not wrap, and a bound like e + 4 <= n must not overflow.  Each case runs one entry point at such a
size with a small exact reference:
  * operands are zero except a few whole images / planes -- the first, the last, and those holding the flat element
    indices 2^30 and total - stride (stride: the grid-stride of a 16-CTA-per-SM grid of 256 threads) --, filled with
    lattice values (integers in [-4, 4], weights +-2^-3 * 2^q), so every output is exact in fp32 and the fp64
    reference runs on the nonzero images only;
  * outputs start as NaN, and the whole output is compared: the reference images bit for bit, zeros elsewhere;
  * where an overrun could stay inside the test's own memory, the tensor is a view into a larger buffer whose 64 words
    on each side hold a pattern that must survive.
At 2^31 elements and beyond, QuantizedConv2d, FusedSyncBatchNorm and optim.SGD hand the call to the stock module.
Each case keeps at most 40 GiB live and releases it before the next."""
import contextlib
import ctypes
import os
import warnings

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = [pytest.mark.gpu, pytest.mark.slow]

import po2_quantization_b200 as P  # noqa: E402
from po2_quantization_b200 import _lib, ops  # noqa: E402
from oracle import po2_oracle as O  # noqa: E402

from tests.test_conv_exact_gpu import lattice_w  # noqa: E402

GUARD = 64
NAN = float("nan")


@pytest.fixture(autouse=True)
def _release():
    """the GPU is shared: each case keeps at most 40 GiB live and releases it"""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    yield
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    print(f"peak {peak / 2**30:.2f} GiB")
    torch.cuda.empty_cache()
    assert peak <= 40 * 2**30, f"{peak / 2**30:.1f} GiB live"


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def grid_stride():
    return torch.cuda.get_device_properties(0).multi_processor_count * 16 * 256


def hot_images(total, per_image):
    """indices of the first and last image and of those holding flat elements 2^30 and total - stride"""
    n_img = total // per_image
    return sorted({min(i, n_img - 1) for i in (0, n_img - 1, (1 << 30) // per_image, (total - grid_stride()) // per_image)})


def lattice(shape, gen):
    return torch.randint(-4, 5, shape, generator=gen, device="cuda").float()


def guarded(n, offset=0):
    """(buffer, view): a float32 view of n elements at `offset` floats after 64 guard words, 64 guard words behind"""
    buf = torch.empty(GUARD + offset + n + GUARD, dtype=torch.float32, device="cuda")
    pattern = torch.arange(GUARD, dtype=torch.int32, device="cuda") | 0x7FA00000          # NaN payloads
    buf[:GUARD + offset].view(torch.int32).copy_(torch.cat([pattern, pattern[:offset]]))
    buf[GUARD + offset + n:].view(torch.int32).copy_(pattern)
    return buf, buf[GUARD + offset:GUARD + offset + n]


def guards_intact(buf, n, offset=0):
    pattern = torch.arange(GUARD, dtype=torch.int32, device="cuda") | 0x7FA00000
    head = buf[:GUARD].view(torch.int32)
    tail = buf[GUARD + offset + n:].view(torch.int32)
    return torch.equal(head, pattern) and torch.equal(tail, pattern)


def all_zero_except(t, images):
    """every element of t (images along dim 0) outside `images` is +-0 -- NaN (never written) fails"""
    keep = [t[i].clone() for i in images]
    for i in images:
        t[i] = 0
    ok = bool(t.eq(0).all())
    for i, v in zip(images, keep):
        t[i] = v
    return ok


@contextlib.contextmanager
def library_path_noted(key_prefix):
    """runs the block with PO2_STRICT off and yields the list of fallback keys noted in it"""
    old = os.environ.pop("PO2_STRICT", None)
    before = set(ops._noted)
    ops._noted.difference_update({k for k in ops._noted if k.startswith(key_prefix)})
    seen = []
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            yield seen
        seen.extend(k for k in ops._noted if k.startswith(key_prefix))
    finally:
        ops._noted.clear()
        ops._noted.update(before)
        if old is not None:
            os.environ["PO2_STRICT"] = old


# ---- depthwise 3x3 (scalar kernels): 576 channels at 7 x 7, B = 76087: 2^31 - 4160 elements on both sides ----------
DW = (76087, 576, 7, 7)
DW_VEC = (65535, 512, 8, 8)                                  # 2^31 - 2^15, the 128-bit kernel


def _dw_operands(seed, shape=DW):
    B, C, H, W = shape
    total = B * C * H * W
    assert total in (2**31 - 4160, 2**31 - 2**15)
    imgs = hot_images(total, C * H * W)
    gen = _gen(seed)
    x = torch.zeros(shape, device="cuda")
    for i in imgs:
        x[i] = lattice((C, H, W), gen)
    w = lattice_w((C, 1, 3, 3), gen)
    return x, w, imgs


@pytest.mark.parametrize("shape", [DW, DW_VEC], ids=["scalar-7x7", "vec-8x8"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_depthwise_forward_just_under_two_to_the_31(dtype, shape):
    """conv_depthwise_kernel (W % 4 != 0) and conv_depthwise_vec_kernel (W % 4 == 0)"""
    B, C, H, W = shape
    x, w, imgs = _dw_operands(1, shape)
    x = x.to(dtype)
    assert ops.conv_kernel_kind(x.shape, w.shape, 1, 1, C, ops.COMPUTE["tf32"], dtype) == 1
    out = torch.full(shape, NAN, dtype=dtype, device="cuda")
    with torch.cuda.device(0):
        ops.conv2d_out(x, w, None, out, 1, 1, C, ops.COMPUTE["tf32"])
    torch.cuda.synchronize()
    ref = F.conv2d(x[imgs].double(), w.double(), None, 1, 1, 1, C).to(dtype)
    assert torch.equal(out[imgs], ref)
    assert all_zero_except(out, imgs)


def test_depthwise_backward_just_under_two_to_the_31():
    """dw_dgrad_kernel and dw_wgrad_kernel: g and x nonzero on the same images"""
    B, C, H, W = DW
    x, w, imgs = _dw_operands(2)
    g = torch.zeros_like(x)
    gen = _gen(3)
    for i in imgs:
        g[i] = lattice((C, H, W), gen)
    lib = _lib.load()
    stream = ops._stream_ptr(x.device)
    gx = torch.full(DW, NAN, device="cuda")
    _lib.check(lib.po2_conv2d_depthwise_dgrad(g.data_ptr(), w.data_ptr(), gx.data_ptr(), B, C, H, W, stream), "dgrad")
    ws = torch.zeros(lib.po2_conv2d_depthwise_wgrad_workspace(C), dtype=torch.uint8, device="cuda")
    gw = torch.full((C, 1, 3, 3), NAN, device="cuda")
    _lib.check(lib.po2_conv2d_depthwise_wgrad(g.data_ptr(), x.data_ptr(), gw.data_ptr(), B, C, H, W, ws.data_ptr(),
                                              ws.numel(), stream), "wgrad")
    torch.cuda.synchronize()
    xd = x[imgs].double().requires_grad_(True)
    wd = w.double().requires_grad_(True)
    F.conv2d(xd, wd, None, 1, 1, 1, C).backward(g[imgs].double())
    assert torch.equal(gx[imgs], xd.grad.float())
    assert all_zero_except(gx, imgs)
    assert torch.equal(gw, wd.grad.float())


def test_dilate2_into_just_under_two_to_the_31():
    """the zero-insertion of a stride-2 backward with odd H (576-channel 7x7 -> 4x4): g_up has 2^31 - 4160 elements"""
    B, C = 76087, 576
    assert B * C * 49 == 2**31 - 4160
    g = torch.randint(-4, 5, (B, C, 4, 4), generator=_gen(4), device="cuda", dtype=torch.int8).float()
    up = torch.full((B, C, 7, 7), NAN, device="cuda")
    with torch.cuda.device(0):
        ops.dilate2_into_out(g, up)
    torch.cuda.synchronize()
    assert torch.equal(up[..., ::2, ::2], g)
    assert bool(up[..., 1::2, :].eq(0).all()) and bool(up[..., ::2, 1::2].eq(0).all())


# ---- BatchNorm at 2^31 - 1024 (scalar path, HW = 49) and 2^31 - 2^14 (VEC path, HW = 1024) --------------------------
BN_SHAPES = [(684784, 64, 7, 7), (131071, 16, 32, 32)]
BN_IDS = ["scalar-7x7", "vec-32x32"]


def _bn_operands(shape, seed, residual):
    B, C, H, W = shape
    total = B * C * H * W
    assert total in (2**31 - 1024, 2**31 - 2**14)
    imgs = hot_images(total, C * H * W)
    gen = _gen(seed)
    x = torch.zeros(shape, device="cuda")
    res = torch.zeros(shape, device="cuda") if residual else None
    for i in imgs:
        x[i] = lattice((C, H, W), gen)
        if residual:
            res[i] = lattice((C, H, W), gen)
    bn = P.FusedSyncBatchNorm(C).cuda()
    with torch.no_grad():
        bn.weight.copy_(torch.linspace(0.5, 1.5, C))
        bn.bias.copy_(torch.linspace(-0.25, 0.25, C))
    return x, res, bn, imgs


def _bn_stats(xs, cnt, eps):
    """fp64 batch statistics in closed form: only the hot images contribute to the sums, the count is B * H * W"""
    mean = xs.sum((0, 2, 3)) / cnt
    var = xs.square().sum((0, 2, 3)) / cnt - mean.square()
    return mean, var, 1.0 / torch.sqrt(var + eps)


def _close(got, ref):
    """the fp32 kernels against fp64: terms of up to ~1000 cancel, so the absolute tolerance is a few fp32 ulps of the
    largest value; a wrong or missing element is off by far more"""
    return torch.allclose(got.double(), ref, rtol=1e-5, atol=4e-6 * (ref.abs().max().item() + 1.0))


def _all_equal_to_one_cold_image(t, imgs):
    """the cold images (zero inputs) all hold the output of the first cold image, bit for bit -- NaN fails"""
    cold = next(i for i in range(t.shape[0]) if i not in imgs)
    const = t[cold].clone()
    keep = [t[i].clone() for i in imgs]
    for i in imgs:
        t[i] = const
    ok = bool(t.eq(const).all())
    for i, v in zip(imgs, keep):
        t[i] = v
    return ok, const


@pytest.mark.parametrize("shape", BN_SHAPES, ids=BN_IDS)
def test_batchnorm_forward_just_under_two_to_the_31(shape):
    """residual + ReLU on the norm kernels (no library path): the hot images against fp64 with the statistics of the
    whole batch, every cold image the per-channel constant relu(beta - mean * gamma * invstd), running statistics"""
    B, C, H, W = shape
    x, res, bn, imgs = _bn_operands(shape, 5, True)
    with library_path_noted("bn:") as seen, torch.no_grad():
        y = bn(x, residual=res, relu=True)
    torch.cuda.synchronize()
    assert not seen, seen
    cnt = B * H * W
    mean, var, invstd = _bn_stats(x[imgs].double(), cnt, bn.eps)
    a = bn.weight.double() * invstd
    b = bn.bias.double() - mean * a
    ref = torch.relu(x[imgs].double() * a.view(1, -1, 1, 1) + b.view(1, -1, 1, 1) + res[imgs].double())
    assert _close(y[imgs], ref)
    assert torch.allclose(bn.running_mean.double(), 0.1 * mean, rtol=1e-5, atol=1e-9)
    assert torch.allclose(bn.running_var.double(), 0.9 + 0.1 * var * cnt / (cnt - 1), rtol=1e-6, atol=1e-9)
    ok, const = _all_equal_to_one_cold_image(y, imgs)
    assert ok
    assert _close(const, torch.relu(b).view(-1, 1, 1).expand(C, H, W))


@pytest.mark.parametrize("shape", BN_SHAPES, ids=BN_IDS)
def test_batchnorm_backward_just_under_two_to_the_31(shape):
    """ReLU backward (reduce + apply kernels) against the closed form: with g = dy masked by y > 0,
    dx = (g - sum g / M - (x - mean) invstd^2 sum g (x - mean) / M) gamma invstd, dgamma, dbeta"""
    B, C, H, W = shape
    x, _, bn, imgs = _bn_operands(shape, 11, False)
    x.requires_grad_(True)
    dy = torch.zeros(shape, device="cuda")
    gen = _gen(12)
    for i in imgs:
        dy[i] = lattice((C, H, W), gen)
    with library_path_noted("bn:") as seen:
        y = bn(x, relu=True)
        y.backward(dy)
    torch.cuda.synchronize()
    assert not seen, seen
    cnt = B * H * W
    xs = x.detach()[imgs].double()
    mean, _, invstd = _bn_stats(xs, cnt, bn.eps)
    v = lambda t: t.view(1, -1, 1, 1)                                   # noqa: E731
    ga = bn.weight.detach().double()
    yh = torch.relu((xs - v(mean)) * v(ga * invstd) + v(bn.bias.detach().double()))
    g = torch.where(yh > 0, dy[imgs].double(), 0.0)
    sg, sgx = g.sum((0, 2, 3)), (g * (xs - v(mean))).sum((0, 2, 3))
    dx_ref = (g - v(sg / cnt) - (xs - v(mean)) * v(invstd.square() * sgx / cnt)) * v(ga * invstd)
    dx = x.grad
    assert _close(dx[imgs], dx_ref)
    assert torch.allclose(bn.bias.grad.double(), sg, rtol=1e-6, atol=1e-6)
    assert torch.allclose(bn.weight.grad.double(), sgx * invstd, rtol=1e-5, atol=1e-5)
    ok, const = _all_equal_to_one_cold_image(dx, imgs)
    assert ok
    cold_ref = (-v(sg / cnt) - (0 - v(mean)) * v(invstd.square() * sgx / cnt)) * v(ga * invstd)
    assert torch.allclose(const.double(), cold_ref[0].expand(C, H, W), rtol=1e-4, atol=1e-9)


# ---- po2_sgd_step: 2^31 - 1 (128-bit path) and 2^31 - 3 at a 4-byte offset (scalar path) ----------------------------
@pytest.mark.parametrize("n, offset", [(2**31 - 1, 0), (2**31 - 3, 1)], ids=["vec-2^31-1", "scalar-2^31-3"])
def test_sgd_step_just_under_two_to_the_31(n, offset):
    """p = 1 everywhere, g zero except a head and a tail slice: torch.optim.SGD's roundings on the slices, p unchanged
    and the momentum buffer zero elsewhere, guard words intact around p, g and the buffer"""
    lr, mom = 0.125, 0.9
    pb, p = guarded(n, offset)
    gb, g = guarded(n, offset)
    bb, buf = guarded(n, offset)
    p.fill_(1.0)
    g.zero_()
    buf.fill_(NAN)
    L = 1 << 16
    gen = _gen(6)
    hs, ts = slice(0, L), slice(n - L, n)
    for s in (hs, ts):
        g[s] = torch.randn(L, generator=gen, device="cuda")
    lib = _lib.load()
    arr = ctypes.c_void_p * 1
    numel = (ctypes.c_longlong * 1)(n)
    for step in range(2):
        _lib.check(lib.po2_sgd_step(arr(p.data_ptr()), arr(g.data_ptr()), arr(buf.data_ptr()), numel, 1, lr, mom, 0.0,
                                    int(step == 0), ops._stream_ptr(p.device)), "po2_sgd_step")
    torch.cuda.synchronize()
    assert guards_intact(pb, n, offset) and guards_intact(gb, n, offset) and guards_intact(bb, n, offset)
    # the stock optimizer on the slices
    ref_p = torch.ones(2 * L, device="cuda", requires_grad=True)
    opt = torch.optim.SGD([ref_p], lr=lr, momentum=mom)
    for _ in range(2):
        ref_p.grad = torch.cat([g[hs], g[ts]])
        opt.step()
    ref_buf = opt.state[ref_p]["momentum_buffer"]
    assert torch.equal(torch.cat([p[hs], p[ts]]), ref_p.detach())
    assert torch.equal(torch.cat([buf[hs], buf[ts]]), ref_buf)
    mid = slice(L, n - L)
    assert bool(p[mid].eq(1.0).all())
    assert bool(buf[mid].eq(0.0).all())


# ---- quantizer: fp32 at 2^31 + 5 and 2^32 + 3, bf16 at 2^32 + 3; fused and two-pass --------------------------------
def _quant_check(x, y, codes, zc, sse, n, zeros, dt):
    """y and codes against the oracle on slices (head, both sides of 2^31 and 2^32, 2^30, the tail holding the maximum),
    the zero count, and sse against an fp64 sum taken in chunks"""
    L = 4096
    starts = [a for a in (0, 2**30 - L // 2, 2**31 - L // 2, 2**32 - L // 2, n - 1 - L) if a + L <= n - 1]
    for a in starts:
        xs = x[a:a + L].float().cpu().numpy()
        ref, q, sgn, _ = O.quantize(np.concatenate([xs, [np.float32(-1.0)]]), 4, 1, False, dtype=dt, return_parts=True)
        got = y[a:a + L].float().cpu().numpy()
        assert np.array_equal(got.view(np.uint32), ref[:L].view(np.uint32)), a
        want = O.pack_codes(O.exponent_codes(q[:L], sgn[:L], 4), 4)
        assert np.array_equal(codes[a // 2:(a + L) // 2].cpu().numpy(), want), a
    last = O.quantize(np.array([x[n - 1].float().item(), -1.0], np.float32), 4, 1, False, dtype=dt)
    assert y[n - 1].float().item() == float(last[0])
    assert zc.item() == len(zeros)
    acc, step = 0.0, 1 << 26
    for a in range(0, n, step):
        acc += float((y[a:a + step].double() - x[a:a + step].double()).square().sum())
    assert abs(sse.item() - acc) <= 1e-4 * acc               # the kernels' per-thread partial sums are fp32
    return starts


@pytest.mark.parametrize("dtype, n", [(torch.float32, 2**31 + 5), (torch.float32, 2**32 + 3), (torch.bfloat16, 2**32 + 3)],
                         ids=["fp32-2^31+5", "fp32-2^32+3", "bf16-2^32+3"])
def test_quantizer_past_two_to_the_31(dtype, n):
    """quantize_full (fused), absmax + quantize (two-pass), dequantize and ste_backward (accumulate) at n > 2^31, with
    zeros planted above 2^31 and 2^32, against the oracle"""
    dt = "f32" if dtype == torch.float32 else "bf16"
    x = torch.empty(n, dtype=dtype, device="cuda")
    gen, step = _gen(7), 1 << 28
    for a in range(0, n, step):                               # +-{1, 2, 3, 4} / 8, generated in chunks
        m = min(step, n - a)
        v = torch.randint(1, 5, (m,), generator=gen, device="cuda", dtype=torch.int8).float().mul_(0.125)
        v.mul_(torch.randint(0, 2, (m,), generator=gen, device="cuda", dtype=torch.int8).float().mul_(2).sub_(1))
        x[a:a + m] = v
        del v
    zeros = [3, 2**31 - 1, 2**31] + ([2**32 - 1, 2**32] if n > 2**32 else []) + [n - 1]
    x[zeros] = 0.0
    assert n - 7 not in zeros
    x[n - 7] = -1.0                                           # the unique maximum of |x|, in the tail slice
    y, codes, scale, zc, sse = torch.ops.po2.quantize_full(x, 4, 1, False)
    torch.cuda.synchronize()
    assert scale.item() == 1.0
    starts = _quant_check(x, y, codes, zc, sse, n, zeros, dt)
    # two passes (po2_absmax, then po2_quantize with that scale) into the same buffers
    y.fill_(NAN)
    codes.fill_(0xA5)
    zc.zero_()
    sse.zero_()
    scale2 = torch.empty((), dtype=torch.float32, device="cuda")
    with torch.cuda.device(0):
        ops.absmax_out(x, scale2)
        ops.quantize_out(x, y, scale2, 4, 1, False, codes, zc, sse)
    torch.cuda.synchronize()
    assert scale2.item() == 1.0
    _quant_check(x, y, codes, zc, sse, n, zeros, dt)
    del x
    torch.cuda.empty_cache()
    d = torch.ops.po2.dequantize(codes, scale, n, 4, 1, dtype)
    # a zero input has no code of its own: it is stored as (+, the smallest level), 2^(fsr - 2^(bits - 1)) = 2^-7
    assert torch.equal(d[zeros].float(), torch.full((len(zeros),), 2.0**-7, device="cuda"))
    d[zeros] = 0.0
    assert torch.equal(d, y)
    del d, codes
    torch.cuda.empty_cache()
    gi = torch.ones(n, dtype=dtype, device="cuda")
    ops.ste_backward(y, gi, True)
    torch.cuda.synchronize()
    for a in starts + [n - 8]:                                # n - 8 .. n - 1: the last element too
        assert torch.equal(gi[a:a + 8], y[a:a + 8] + 1.0), a


# ---- tensor cores: 16 -> 16 3x3 pad 1 at 32 x 32, B = 131071: 2^31 - 2^14 elements on both sides ----------------------
TC = (131071, 16, 32, 32)


def _fwd_ep(x, w, out, a, b, res, act, compute):
    """po2_conv2d_fwd_ep_dt into a caller-made (NaN-filled) output: act(conv(x, w) * a[k] + b[k] + res)"""
    lib = _lib.load()
    B, C, H, W = x.shape
    K = w.shape[0]
    dt = 1 if x.dtype == torch.bfloat16 else 0
    need = lib.po2_conv2d_workspace_dt(B, C, H, W, K, 3, 3, 1, 1, 1, compute, dt)
    ws = torch.empty(max(int(need), 16), dtype=torch.uint8, device="cuda")
    _lib.check(lib.po2_conv2d_fwd_ep_dt(x.data_ptr(), w.data_ptr(), None, out.data_ptr(), B, C, H, W, K, 3, 3, 1, 1, 1,
                                        _lib.W_F32_PO2, 4, 1, compute, ws.data_ptr(), ws.numel(), a.data_ptr(),
                                        b.data_ptr(), res.data_ptr(), act, dt, ops._stream_ptr(x.device)),
               "po2_conv2d_fwd_ep_dt")


@pytest.mark.parametrize("compute, dtype, kind, wkind", [(2, torch.float32, 3, 2), (0, torch.float32, 2, 1),
                                                         (2, torch.bfloat16, 2, None)],
                         ids=["k3t-k5t-tf32", "k3-k5-bf16ops", "k3-bf16x"])
def test_tensor_core_conv_just_under_two_to_the_31(compute, dtype, kind, wkind):
    """the forward with the folded epilogue, residual and ReLU (K3T / K3, and K3 on a bf16 x at inference), the data
    gradient (same kernel) and the weight gradient (K5T / K5), bit for bit on sparse lattice operands"""
    B, C, H, W = TC
    total = B * C * H * W
    assert total == 2**31 - 2**14
    imgs = hot_images(total, C * H * W)
    lib = _lib.load()
    assert lib.po2_conv2d_kernel_kind_dt(B, C, H, W, C, 3, 3, 1, 1, 1, compute, 1 if dtype == torch.bfloat16 else 0) \
        == kind
    gen = _gen(20 + compute)
    w = lattice_w((C, C, 3, 3), gen)
    a = torch.exp2(torch.randint(-2, 3, (C,), generator=gen, device="cuda").float())
    a = a * (torch.randint(0, 2, (C,), generator=gen, device="cuda").float() * 2 - 1)
    b = torch.randint(-512, 513, (C,), generator=gen, device="cuda").float() * 2.0 ** -8
    x = torch.zeros(TC, dtype=dtype, device="cuda")
    res = torch.zeros(TC, dtype=dtype, device="cuda")
    for i in imgs:
        x[i] = lattice((C, H, W), gen)
        res[i] = lattice((C, H, W), gen)
    out = torch.full(TC, NAN, dtype=dtype, device="cuda")
    _fwd_ep(x, w, out, a, b, res, 1, compute)
    torch.cuda.synchronize()
    v = lambda t: t.double().view(1, -1, 1, 1)                          # noqa: E731
    pre = F.conv2d(x[imgs].double(), w.double(), None, 1, 1) * v(a) + v(b) + res[imgs].double()
    assert pre.abs().max().item() < 2**12                   # a multiple of 2^-12: exact in fp32
    assert torch.equal(out[imgs], torch.relu(pre).to(dtype))
    ok, const = _all_equal_to_one_cold_image(out, imgs)     # the cold images: relu(b[k])
    assert ok and torch.equal(const, torch.relu(b).to(dtype).view(-1, 1, 1).expand(C, H, W))
    del out, res
    if wkind is None:                                        # bf16: inference only
        return
    g = torch.zeros(TC, device="cuda")
    for i in imgs:
        g[i] = lattice((C, H, W), gen)
    gx = torch.full(TC, NAN, device="cuda")
    scale = torch.tensor(2.0 ** -3, device="cuda")
    assert ops.conv2d_dgrad_out(g, w, scale, gx, 1, compute)
    torch.cuda.synchronize()
    ref = torch.nn.grad.conv2d_input((len(imgs), C, H, W), w.double(), g[imgs].double(), padding=1).float()
    assert torch.equal(gx[imgs], ref)
    assert all_zero_except(gx, imgs)
    del gx
    assert lib.po2_conv2d_wgrad_kernel_kind(B, C, H, W, C, 3, 3, 1, 1, 1, compute) == wkind
    gw = torch.full((C, C, 3, 3), NAN, device="cuda")
    assert ops.conv2d_wgrad_out(g, x, gw, 1, compute)
    torch.cuda.synchronize()
    ref = torch.nn.grad.conv2d_weight(x[imgs].double(), (C, C, 3, 3), g[imgs].double(), padding=1).float()
    assert torch.equal(gw, ref)


def test_stride2_backward_with_a_two_to_the_31_zero_inserted_gradient_runs_aten():
    """16 -> 32 3x3 stride 2 at 32 x 32, B = 65536: x has 2^30 elements and the forward runs on K3, but the zero-inserted
    output gradient (B, 32, 32, 32) would have 2^31.  The backward leaves the kernels before dilating, reported, and
    equals nn.Conv2d's on the quantized weight"""
    B = 65536
    lib = _lib.load()
    assert lib.po2_conv2d_kernel_kind(B, 16, 32, 32, 32, 3, 3, 2, 1, 1, 2) in (2, 3)
    conv = P.QuantizedConv2d(16, 32, 3, stride=2, padding=1, quantize_fn=P.PowerOfTwoQuantizer, bits=4).cuda()
    gen = _gen(30)
    with torch.no_grad():
        conv.weight.copy_(lattice_w((32, 16, 3, 3), gen))
    x = torch.zeros(B, 16, 32, 32, device="cuda")
    g = torch.zeros(B, 32, 16, 16, device="cuda")
    imgs = hot_images(x.numel(), 16 * 32 * 32)
    for i in imgs:
        x[i] = lattice((16, 32, 32), gen)
        g[i] = lattice((32, 16, 16), gen)
    x.requires_grad_(True)
    with library_path_noted("conv_backward_aten") as seen:
        out = conv(x)
        out.backward(g)
    torch.cuda.synchronize()
    assert seen, "the fallback was not reported"
    del out
    qw = P.PowerOfTwoQuantizer.apply(conv.weight.detach(), 4)
    xh = x.detach()[imgs].double().requires_grad_(True)
    wd = qw.double().requires_grad_(True)
    F.conv2d(xh, wd, None, 2, 1).backward(g[imgs].double())
    assert torch.allclose(x.grad[imgs].double(), xh.grad, rtol=1e-3, atol=1e-3)
    assert all_zero_except(x.grad, imgs)
    assert torch.allclose(conv.weight.grad.double(), wd.grad, rtol=1e-3, atol=1e-3)


# ---- just over the bound: the drop-in classes hand the call to the stock modules -------------------------------------
def test_quantized_conv2d_at_two_to_the_31_runs_nn_conv2d():
    """16->16 3x3 at 32 x 32, B = 131072: x and the output have 2^31 elements.  QuantizedConv2d equals nn.Conv2d on the
    quantized weight, with the fallback reported"""
    B = 131072
    conv = P.QuantizedConv2d(16, 16, 3, stride=1, padding=1, quantize_fn=P.PowerOfTwoQuantizer, bits=4).cuda()
    gen = _gen(8)
    x = torch.zeros(B, 16, 32, 32, device="cuda")
    imgs = hot_images(x.numel(), 16 * 32 * 32)
    for i in imgs:
        x[i] = lattice((16, 32, 32), gen)
    with torch.no_grad():
        conv.weight.copy_(lattice_w((16, 16, 3, 3), gen))
    with library_path_noted("qconv:") as seen, torch.no_grad():
        out = conv(x)
    assert seen, "the size fallback was not reported"
    ref_conv = nn.Conv2d(16, 16, 3, 1, 1, bias=False).cuda()
    with torch.no_grad():
        ref_conv.weight.copy_(P.PowerOfTwoQuantizer.apply(conv.weight, 4))
        ref = ref_conv(x[imgs])                               # the other images are zero, and so is their output
    del x
    assert torch.allclose(out[imgs], ref, rtol=1e-3, atol=1e-3)
    assert all_zero_except(out, imgs)


def test_fused_batchnorm_at_two_to_the_31_runs_nn_batchnorm():
    shape = (65536, 32, 32, 32)                               # 2^31 elements
    gen = _gen(9)
    x = torch.zeros(shape, device="cuda")
    for i in hot_images(x.numel(), 32 * 32 * 32):
        x[i] = lattice(shape[1:], gen)
    bn = P.FusedSyncBatchNorm(32).cuda()
    ref_bn = nn.BatchNorm2d(32).cuda()
    with library_path_noted("bn:") as seen, torch.no_grad():
        y = bn(x)
    assert seen, "the size fallback was not reported"
    with torch.no_grad():
        ref = ref_bn(x)
    assert torch.equal(y, ref)
    assert torch.equal(bn.running_mean, ref_bn.running_mean) and torch.equal(bn.running_var, ref_bn.running_var)


def test_sgd_at_two_to_the_31_runs_torch_sgd():
    """a 2^31-element parameter beside a small one: optim.SGD equals torch.optim.SGD on both"""
    n = 2**31
    gen = _gen(10)
    big = torch.zeros(n, device="cuda")
    big[:4096] = 1.0
    big[-4096:] = 2.0
    small = torch.randn(1000, generator=gen, device="cuda")
    gbig = torch.zeros(n, device="cuda")
    gbig[:4096] = torch.randn(4096, generator=gen, device="cuda")
    gbig[-4096:] = torch.randn(4096, generator=gen, device="cuda")
    gsmall = torch.randn(1000, generator=gen, device="cuda")
    pb, ps = nn.Parameter(big), nn.Parameter(small.clone())
    pb.grad, ps.grad = gbig, gsmall
    opt = P.optim.SGD([pb, ps], lr=0.1, momentum=0.9)
    with library_path_noted("sgd:") as seen:
        opt.step()
    assert seen, "the size fallback was not reported"
    head, tail = pb.detach()[:8192].clone(), pb.detach()[-8192:].clone()
    mid_ok = bool(pb.detach()[4096:-4096].eq(0).all())
    del pb, big
    torch.cuda.empty_cache()
    # the stock optimizer on the nonzero slices of the big parameter and on the small one
    rb = nn.Parameter(torch.cat([torch.ones(4096, device="cuda"), torch.zeros(4096, device="cuda"),
                                 torch.zeros(4096, device="cuda"), torch.full((4096,), 2.0, device="cuda")]))
    rb.grad = torch.cat([gbig[:4096], torch.zeros(8192, device="cuda"), gbig[-4096:]])
    rs = nn.Parameter(small.clone())
    rs.grad = gsmall
    torch.optim.SGD([rb, rs], lr=0.1, momentum=0.9).step()
    assert torch.equal(torch.cat([head, tail]), rb.detach())
    assert torch.equal(ps.detach(), rs.detach())
    assert mid_ok
