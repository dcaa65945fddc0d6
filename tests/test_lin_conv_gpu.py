"""lin / lin+ layers on the sm_100a conv kernels (utils/quantizers.py:59-136 + models/quantized_conv.py:32-38).

After at least one refinement round a lin weight is n * 2^k per input channel with |n| <= 2^(bits-1) - 1, so it is
its own exact tensor-core operand (bf16 up to 9 bits, tf32 up to 12) and runs with scale 1.0 through every consumer
of (packed, scale).  These tests hold the quantizer bit-identical to po2_lin_quantize, the operand exact, the QAT and
PTQ layers, the prefetch and the training step to the stock path within the tolerances the PO2 layers are held to."""
import collections
import copy

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import po2_quantization_b200 as P  # noqa: E402
from po2_quantization_b200 import _lib, ops  # noqa: E402
from tests.test_conv_gpu import ALL, MOBILENET, ODD, RESNET, TOL_FP32, TOL_TC, TOL_TF32  # noqa: E402

LIN = [(P.LinearPowerOfTwoQuantizer, False), (P.LinearPowerOfTwoPlusQuantizer, True)]
LIN_IDS = ["lin", "lin+"]
BITS = (2, 4, 8)
TOL = {0: TOL_TC, 1: TOL_FP32, 2: TOL_TF32}


def _case(case, seed=0):
    name, B, C, H, W, K, k, stride, pad, groups = case
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(B, C, H, W, device="cuda", generator=g)
    w = torch.randn(K, C // groups, k, k, device="cuda", generator=g) * 0.1
    return x, w


def _bits_eq(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _rel(out, ref):
    return ((out.double() - ref).abs().max() / ref.abs().max()).item()


def _quantize_pack(w, xshape, stride, pad, groups, bits, plus, compute):
    """(y, packed) from po2_lin_quantize_pack, or None when the geometry has no tensor-core operand"""
    lib = _lib.load()
    B, C, H, W_ = xshape
    K, _, R, S = w.shape
    nbytes = int(lib.po2_conv2d_pack_bytes(B, C, H, W_, K, R, S, stride, pad, groups, compute))
    if nbytes == 0:
        return None
    y = torch.empty_like(w)
    packed = torch.empty(nbytes, dtype=torch.uint8, device=w.device)
    _lib.check(lib.po2_lin_quantize_pack(w.data_ptr(), y.data_ptr(), packed.data_ptr(), nbytes, None, 0, B, C, H, W_, K,
                                         R, S, stride, pad, groups, bits, 10, int(plus), ops._flavor, compute,
                                         ops._stream_ptr(w.device)), "po2_lin_quantize_pack")
    return y, packed


# ---- 1. the quantizer is bit-identical to po2_lin_quantize ---------------------------------------------------------
@pytest.mark.parametrize("compute", [0, 2], ids=["bf16", "tf32"])
@pytest.mark.parametrize("q", LIN, ids=LIN_IDS)
@pytest.mark.parametrize("case", ALL, ids=[c[0] for c in ALL])
def test_lin_quantize_pack_y_is_bit_identical(case, q, compute):
    cls, plus = q
    name, B, C, H, W, K, k, stride, pad, groups = case
    x, w = _case(case)
    for bits in BITS:
        want = cls.forward(None, w, bits=bits)
        got = _quantize_pack(w, x.shape, stride, pad, groups, bits, plus, compute)
        if got is None:
            continue
        assert _bits_eq(got[0], want), (name, bits)


@pytest.mark.parametrize("compute", [0, 2], ids=["bf16", "tf32"])
@pytest.mark.parametrize("q", LIN, ids=LIN_IDS)
def test_lin_multi_tensor_launch_y_is_bit_identical(q, compute):
    """one launch over every shape of the tables (random weights) and the reference's golden vectors"""
    cls, plus = q
    from tests import golden_util as G
    lib = _lib.load()
    z = G.load("lin_golden.npz")
    tensors = [(w, x.shape, c[7], c[8], c[9]) for c in ALL for x, w in [_case(c, seed=3)]]
    tensors.append((torch.from_numpy(z["w"]).cuda(), (8, 16, 16, 16), 1, 1, 1))
    for bits in BITS:
        dbytes = int(lib.po2_lin_multi_desc_bytes())
        host = torch.zeros(len(tensors) * dbytes, dtype=torch.uint8)
        taken, ctas, elems, keep = [], 0, 1, []
        for w, xs, stride, pad, groups in tensors:
            B, C, H, W_ = xs
            K, _, R, S = w.shape
            nbytes = int(lib.po2_conv2d_pack_bytes(B, C, H, W_, K, R, S, stride, pad, groups, compute))
            if nbytes == 0:
                continue
            y = torch.full_like(w, float("nan"))
            packed = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
            rc = lib.po2_lin_multi_desc_fill(host.data_ptr(), len(taken), w.data_ptr(), y.data_ptr(), packed.data_ptr(),
                                             nbytes, None, 0, B, C, H, W_, K, R, S, stride, pad, groups, bits, 10,
                                             int(plus), ops._flavor, compute)
            if rc == -10:
                continue
            assert rc == C, rc
            taken.append((w, y))
            keep.append(packed)
            ctas += rc
            elems = max(elems, K * R * S)
        assert len(taken) >= 10
        dev = host[:len(taken) * dbytes].cuda()
        _lib.check(lib.po2_lin_quantize_pack_multi(dev.data_ptr(), len(taken), ctas, elems, ops._stream_ptr(dev.device)),
                   "po2_lin_quantize_pack_multi")
        torch.cuda.synchronize()
        for i, (w, y) in enumerate(taken):
            assert _bits_eq(y, cls.forward(None, w, bits=bits)), (bits, i)
    for bits in (3, 4):                                   # the golden vectors through the packing kernel
        name = "lin+" if plus else "lin"
        y, _packed = _quantize_pack(torch.from_numpy(z["w"]).cuda(), (8, 16, 16, 16), 1, 1, 1, bits, plus, compute)
        assert np.array_equal(y.cpu().numpy().view(np.uint32), z[f"{name}|{bits}"].view(np.uint32)), (name, bits)


# ---- 2. the operand is exact -------------------------------------------------------------------------------------
def _round_operand(x, compute):
    if compute == 0:
        return x.bfloat16().float()
    return (x.view(torch.int32) & ~0x1FFF).view(torch.float32)


@pytest.mark.parametrize("compute", [0, 1, 2], ids=["bf16", "fp32", "tf32"])
@pytest.mark.parametrize("q", LIN, ids=LIN_IDS)
@pytest.mark.parametrize("case", ALL, ids=[c[0] for c in ALL])
def test_lin_conv_operand_is_exact(case, q, compute):
    cls, plus = q
    name, B, C, H, W, K, k, stride, pad, groups = case
    x, w = _case(case, seed=1)
    for bits in BITS:
        out, y = ops.lin_qconv2d(x, w, bits, plus, stride, pad, groups, compute)
        assert _bits_eq(y, cls.forward(None, w, bits=bits))
        ref = F.conv2d(x.double(), y.double(), None, stride, pad, 1, groups)
        assert _rel(out, ref) <= TOL[compute], (name, bits, _rel(out, ref))
        if compute == 1:
            continue                                  # fp32 FMA: held to TOL_FP32 above
        # activations already on the operand grid: only fp32 summation error is left
        xr = _round_operand(x, compute)
        out, _ = ops.lin_qconv2d(xr, w, bits, plus, stride, pad, groups, compute)
        ref = F.conv2d(xr.double(), y.double(), None, stride, pad, 1, groups)
        assert _rel(out, ref) <= 1e-6, (name, bits, _rel(out, ref))


# ---- 3. the QAT layer ------------------------------------------------------------------------------------------------
QAT_CASES = [c for c in RESNET + MOBILENET if c[0] in ("r_16_16_3s1", "r_16_32_3s2", "r_16_32_1s2", "m_dw_96_s2",
                                                        "m_pw_576_160", "m_pw_144_32")]


@pytest.mark.parametrize("mode", ["tc", "tf32"])
@pytest.mark.parametrize("q", LIN, ids=LIN_IDS)
@pytest.mark.parametrize("case", QAT_CASES, ids=[c[0] for c in QAT_CASES])
def test_lin_qat_layer_forward_and_gradients(case, q, mode, monkeypatch):
    cls, plus = q
    name, B, C, H, W, K, k, stride, pad, groups = case
    noted = []
    monkeypatch.setattr(ops, "note_library_path", lambda key, msg: noted.append(key))
    ops.set_conv_mode(mode)
    try:
        for bits in BITS:
            x, w = _case(case, seed=bits)
            conv = P.QuantizedConv2d(C, K, k, stride=stride, padding=pad, groups=groups, quantize_fn=cls, bits=bits).cuda()
            with torch.no_grad():
                conv.weight.copy_(w)
            xa = x.clone().requires_grad_(True)
            out = conv(xa)
            gout = torch.randn_like(out)
            out.backward(gout)
            y = cls.forward(None, w, bits=bits).double().requires_grad_(True)
            xd = x.double().requires_grad_(True)
            ref = F.conv2d(xd, y, None, stride, pad, 1, groups)
            ref.backward(gout.double())
            tol = TOL[ops.COMPUTE[mode]]
            assert _rel(out.detach(), ref.detach()) <= tol, (name, bits)
            assert _rel(xa.grad, xd.grad) <= TOL_TC, (name, bits)
            assert _rel(conv.weight.grad, y.grad) <= TOL_TC, (name, bits)          # straight-through into the master
        assert not [k for k in noted if k.startswith(("qconv:", "lin:"))], noted   # the forward ran on our kernels
    finally:
        ops.set_conv_mode(ops.DEFAULT_CONV_MODE)


# ---- 4. the multi-tensor prefetch ------------------------------------------------------------------------------------
@pytest.mark.parametrize("q", LIN, ids=LIN_IDS)
def test_lin_weight_prefetch_equals_inline_quantization(q):
    cls, plus = q
    from workloads import resnet_cifar
    torch.manual_seed(12)
    torch.backends.cudnn.deterministic = True
    try:
        a = resnet_cifar(20, 10, cls, 4).cuda().train()
        b = copy.deepcopy(a)
        P.enable_weight_prefetch(b)
        oa = torch.optim.SGD(a.parameters(), lr=0.05, momentum=0.9)
        ob = torch.optim.SGD(b.parameters(), lr=0.05, momentum=0.9)
        x = torch.randn(32, 3, 32, 32, device="cuda")
        t = torch.randint(0, 10, (32,), device="cuda")
        for it in range(3):
            for m, o in ((a, oa), (b, ob)):
                o.zero_grad()
                F.cross_entropy(m(x), t).backward()
                o.step()
            used = sum(1 for m in b.modules() if getattr(m, "_po2_prefetch", None))
            assert (used > 0) == (it > 0), (it, used)
            for (n, pa), pb in zip(a.named_parameters(), b.parameters()):
                assert torch.equal(pa, pb), (it, n)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            xs = x.clone()

            def step(m, o):
                o.zero_grad()
                F.cross_entropy(m(xs), t).backward()
                o.step()
            step(b, ob), step(a, oa)
            torch.cuda.current_stream().synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                step(b, ob)
            for _ in range(2):
                g.replay()
                step(a, oa)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        for (n, pa), pb in zip(a.named_parameters(), b.parameters()):
            assert torch.equal(pa, pb), ("graph", n)
    finally:
        torch.backends.cudnn.deterministic = False


@pytest.mark.parametrize("q", LIN, ids=LIN_IDS)
def test_lin_weights_are_requantized_after_the_multi_tensor_sgd_step(q):
    cls, plus = q
    from workloads import resnet_cifar
    torch.manual_seed(4)
    dev = torch.device("cuda:0")
    model = resnet_cifar(20, 10, cls, 4).to(dev).train()
    P.enable_weight_prefetch(model)
    opt = P.optim.SGD(model.parameters(), lr=0.5, momentum=0.9, weight_decay=1e-4)
    x = torch.randn(32, 3, 32, 32, device=dev)
    y = torch.randint(0, 10, (32,), device=dev)
    crit = nn.CrossEntropyLoss()
    conv = [m for m in model.modules() if isinstance(m, P.QuantizedConv2d)][3]

    def step():
        opt.zero_grad(set_to_none=True)
        crit(model(x), y).backward()
        opt.step()

    for _ in range(3):
        step()
        model(x)
        torch.cuda.synchronize()
        assert torch.equal(conv.__dict__["_po2_prefetch"].qw, cls.forward(None, conv.weight.detach(), bits=4))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            step()
        s.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            step()
        before = conv.weight.detach().clone()
        for _ in range(2):
            g.replay()
        s.synchronize()
        assert not torch.equal(before, conv.weight)
    torch.cuda.current_stream().wait_stream(s)
    w_before_last = conv.weight.detach().clone()
    with torch.cuda.stream(s):
        g.replay()
        s.synchronize()
    torch.cuda.synchronize()
    assert torch.equal(conv.__dict__["_po2_prefetch"].qw, cls.forward(None, w_before_last, bits=4))


# ---- 5. the launch list of the training step --------------------------------------------------------------------------
def _step_kernels(quantize_fn):
    """kernel names of one eager ResNet-56 4-bit QAT step built as bench.build_training builds it"""
    from torch.profiler import ProfilerActivity, profile
    from workloads import resnet_cifar
    torch.manual_seed(8)
    dev = torch.device("cuda:0")
    model = resnet_cifar(56, 10, quantize_fn, 4).to(dev).train()
    P.enable_weight_prefetch(model)
    opt = P.optim.SGD(model.parameters(), lr=0.1, momentum=0.9, weight_decay=1e-4)
    crit = nn.CrossEntropyLoss()
    x = torch.randn(128, 3, 32, 32, device=dev)
    t = torch.randint(0, 10, (128,), device=dev)

    def step():
        opt.zero_grad(set_to_none=True)
        crit(model(x), t).backward()
        opt.step()

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    return collections.Counter(e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                               and not e.name.startswith(("Memcpy", "Memset")))


@pytest.mark.parametrize("q", LIN, ids=LIN_IDS)
def test_lin_qat_step_launch_list_is_the_po2_list(q, monkeypatch):
    cls, plus = q
    monkeypatch.setenv("PO2_STRICT", "1")
    old = ops.get_wgrad_overlap()
    ops.set_wgrad_overlap(True)
    try:
        po2 = _step_kernels(P.PowerOfTwoQuantizer)
        lin = _step_kernels(cls)
    finally:
        ops.set_wgrad_overlap(old)
    po2_multi = [n for n in po2 if "multi_fused_kernel" in n]
    lin_multi = [n for n in lin if "lin_multi_kernel" in n]
    assert len(po2_multi) == 1 and po2[po2_multi[0]] == 1, po2_multi
    assert len(lin_multi) == 1 and lin[lin_multi[0]] == 1, lin_multi
    want = po2.copy()
    del want[po2_multi[0]]
    want[lin_multi[0]] = 1
    assert lin == want, (lin - want, want - lin)
    assert not [n for n in lin if "lin_quantize_kernel" in n]                      # no per-layer lin launch
    cudnn = [n for n in lin if "cudnn" in n.lower() or "xmma" in n.lower() or "implicit_gemm" in n.lower()]
    assert sum(lin[n] for n in cudnn) == sum(po2[n] for n in cudnn)


# ---- 6. post-training quantization ---------------------------------------------------------------------------------
def _eval_models():
    from workloads import mobilenet_v2_cifar, resnet_cifar
    torch.manual_seed(3)
    return {"resnet20": resnet_cifar(20, 10, None, 4), "mobilenetv2": mobilenet_v2_cifar(10, None, 4)}


@pytest.mark.parametrize("q", LIN, ids=LIN_IDS)
def test_lin_ptq_eval_forward_fold_graph_deepcopy_and_checkpoint(q, monkeypatch):
    cls, plus = q
    x = torch.randn(64, 3, 32, 32, device="cuda")
    for name, model in _eval_models().items():
        model = model.cuda()
        ref_model = copy.deepcopy(model)
        mse = P.quantize_model(model, cls, 4)
        # the returned MSE is the reference's fp32 sum, unchanged
        total, n = None, 0
        with torch.no_grad():
            for m in ref_model.modules():
                if isinstance(m, P.QuantizedConv2d):
                    for p in m.parameters():
                        qp = cls.forward(None, p, bits=4)
                        e = torch.sum((qp - p) ** 2).double()
                        total = e if total is None else total + e
                        n += p.numel()
        assert mse == float((total / n).item())
        tagged = [m for m in model.modules() if isinstance(m, P.QuantizedConv2d) and "_po2_lin_ptq" in m.__dict__]
        assert tagged
        # train-mode passes to give the norms non-trivial running statistics, then evaluate against the stock conv
        # in true fp32.  The bound is the one the PO2 PTQ models are held to on the tcgen05 path (tf32 activations
        # through every layer of the model; each layer alone is within TOL_TF32, test_lin_conv_operand_is_exact),
        # and the fp32-accumulate mode's bound for the CUDA-core kernels
        old_tf32 = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = False
        try:
            with torch.no_grad():
                model.train()
                ops.set_conv_mode("cudnn")
                for _ in range(3):
                    model(torch.randn(64, 3, 32, 32, device="cuda"))
                model.eval()
                want = model(x).double()
                monkeypatch.setenv("PO2_STRICT", "1")
                for mode, tol in (("tf32", 1e-2), ("fp32", 1e-4)):
                    ops.set_conv_mode(mode)
                    for fold in (False, True):
                        m = copy.deepcopy(model)                      # the copy keeps the packed path
                        assert all(c.__dict__.get("_po2_lin_ptq", (None,))[0] == c.weight._version
                                   for c in m.modules() if isinstance(c, P.QuantizedConv2d) and "_po2_lin_ptq" in c.__dict__)
                        if fold:
                            assert P.fold_conv_bn(m) > 0
                        eager = m(x)
                        assert _rel(eager, want) <= tol, (name, mode, fold, _rel(eager, want))
                        assert torch.equal(eager.argmax(1), want.argmax(1)) or mode == "tf32"
                        if mode == "tf32":
                            assert any(c.__dict__.get("_po2_pack_cache") for c in m.modules()
                                       if isinstance(c, P.QuantizedConv2d))
                        s = torch.cuda.Stream()
                        s.wait_stream(torch.cuda.current_stream())
                        with torch.cuda.stream(s):
                            m(x)
                            s.synchronize()
                            g = torch.cuda.CUDAGraph()
                            with torch.cuda.graph(g, stream=s):
                                out = m(x)
                            g.replay()
                            s.synchronize()
                        torch.cuda.current_stream().wait_stream(s)
                        assert torch.equal(out, eager), (name, mode, fold)
                monkeypatch.delenv("PO2_STRICT")
        finally:
            torch.backends.cudnn.allow_tf32 = old_tf32
            ops.set_conv_mode(ops.DEFAULT_CONV_MODE)
        packed = P.pack_state_dict(model)
        assert packed["meta"]["raw_fallbacks"] == [] and not packed["packed"]
        back = P.unpack_state_dict(packed)
        sd = model.state_dict()
        assert list(back) == list(sd)
        for k, v in sd.items():
            assert torch.equal(back[k], v) and back[k].dtype == v.dtype, k
    ops.set_conv_mode(ops.DEFAULT_CONV_MODE)


# ---- 7. edge cases -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("compute", [0, 1, 2], ids=["bf16", "fp32", "tf32"])
def test_lin_nan_and_constant_channels_give_nonfinite_outputs_where_fp64_does(compute):
    for case in (RESNET[0], MOBILENET[9], ODD[1]):
        name, B, C, H, W, K, k, stride, pad, groups = case
        x, w = _case(case, seed=5)
        for bad in ("nan", "const"):
            wb = w.clone()
            if bad == "nan":
                wb[0, 0, 0, 0] = float("nan")
            else:
                wb[:, 0] = 0.25
            out, y = ops.lin_qconv2d(x, wb, 4, False, stride, pad, groups, compute)
            ref = F.conv2d(x.double(), y.double(), None, stride, pad, 1, groups)
            assert not torch.isfinite(ref).all()
            assert torch.equal(torch.isfinite(out), torch.isfinite(ref)), (name, bad)


@pytest.mark.parametrize("mode,bits", [("tc", 10), ("tf32", 13)])
@pytest.mark.parametrize("q", LIN, ids=LIN_IDS)
def test_lin_bits_beyond_the_exact_operand_take_the_library_path(mode, bits, q, monkeypatch):
    cls, plus = q
    noted = []
    monkeypatch.setattr(ops, "note_library_path", lambda key, msg: noted.append(key))
    torch.backends.cudnn.deterministic = True
    ops.set_conv_mode(mode)
    try:
        case = RESNET[0]
        name, B, C, H, W, K, k, stride, pad, groups = case
        x, w = _case(case)
        conv = P.QuantizedConv2d(C, K, k, stride=stride, padding=pad, quantize_fn=cls, bits=bits).cuda()
        with torch.no_grad():
            conv.weight.copy_(w)
        out = conv(x)
        assert any(key.startswith("qconv:lin weights of") for key in noted), noted
        want = F.conv2d(x, cls.apply(w, bits), None, stride, pad)
        assert torch.equal(out, want)
        # the PTQ form of the same layer: reported, the stock conv of the quantized weight
        noted.clear()
        ptq = P.QuantizedConv2d(C, K, k, stride=stride, padding=pad).cuda()
        with torch.no_grad():
            ptq.weight.copy_(w)
        P.quantize_model(ptq, cls, bits)
        with torch.no_grad():
            out = ptq(x)
        assert any(key.startswith("qconv:lin weights of") for key in noted), noted
        assert torch.equal(out, F.conv2d(x, ptq.weight, None, stride, pad))
    finally:
        ops.set_conv_mode(ops.DEFAULT_CONV_MODE)
        torch.backends.cudnn.deterministic = False


# ---- 8. training tracks the stock path -----------------------------------------------------------------------------
def test_lin_plus_qat_loss_curve_tracks_the_stock_path():
    from tests.test_models_gpu import _learnable_batches, _smooth, _train_curve
    from workloads import resnet_cifar
    steps = 50
    batches = [(x.cuda(), y.cuda()) for x, y in _learnable_batches()]
    torch.manual_seed(8)
    init = resnet_cifar(20, 10, P.LinearPowerOfTwoPlusQuantizer, 4).state_dict()
    curves = {}
    old_tf32 = torch.backends.cudnn.allow_tf32
    try:
        ops.set_conv_mode("cudnn")
        for name, tf32 in (("stock_fp32", False), ("stock_tf32_default", True)):
            torch.backends.cudnn.allow_tf32 = tf32
            m = resnet_cifar(20, 10, P.LinearPowerOfTwoPlusQuantizer, 4)
            m.load_state_dict(init)
            curves[name] = _train_curve(m.cuda().train(), batches, steps)
        torch.backends.cudnn.allow_tf32 = False
        for name, mode in (("lin_plus_bf16_operands", "tc"), ("lin_plus_tf32_operands", "tf32")):
            ops.set_conv_mode(mode)
            m = resnet_cifar(20, 10, P.LinearPowerOfTwoPlusQuantizer, 4)
            m.load_state_dict(init)
            curves[name] = _train_curve(m.cuda().train(), batches, steps)
    finally:
        torch.backends.cudnn.allow_tf32 = old_tf32
        ops.set_conv_mode(ops.DEFAULT_CONV_MODE)
    ref = _smooth(curves["stock_fp32"])
    band = {k: max(abs(a - b) for a, b in zip(_smooth(v), ref)) for k, v in curves.items()}
    final = {k: sum(v[-10:]) / 10 for k, v in curves.items()}
    assert final["stock_fp32"] < 0.8 * curves["stock_fp32"][0], "the stock path itself did not learn"
    allowed = max(2.0 * band["stock_tf32_default"], 0.08 * curves["stock_fp32"][0])
    for k in ("lin_plus_bf16_operands", "lin_plus_tf32_operands"):
        assert band[k] <= allowed, (k, band[k], allowed, band)
        assert abs(final[k] - final["stock_fp32"]) <= 0.15 * curves["stock_fp32"][0], (k, final)
        assert final[k] < 0.8 * curves[k][0], (k, "did not learn", final[k], curves[k][0])
