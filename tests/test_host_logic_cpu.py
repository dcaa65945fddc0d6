"""CPU tests of the host-side mirror: API surface, lin/lin+ parity with reference vectors, and the
quantize_model / QuantizedConv2d control flow driven through a fake backend (the oracle) so that no
GPU is needed.  The kernels themselves are covered by the -m gpu suite."""
import copy
import inspect

import numpy as np
import pytest
import torch

import po2_quantization_b200 as P
from po2_quantization_b200 import ops
from tests import golden_util as G


def test_public_surface_matches_reference_names():
    assert list(P.quantizer_dict) == ["lin", "lin+", "po2", "po2+"]          # utils/quantizers.py:156-161
    for cls in P.quantizer_dict.values():
        assert issubclass(cls, torch.autograd.Function)
        assert list(inspect.signature(cls.forward).parameters)[:3] == ["ctx", "input", "bits"]
    sig = inspect.signature(P.QuantizedConv2d.__init__)
    assert [p for p in sig.parameters][1:] == ["in_channels", "out_channels", "kernel_size", "stride", "padding",
                                               "dilation", "groups", "bias", "quantize_fn", "bits"]
    assert sig.parameters["padding"].default == 1 and sig.parameters["bias"].default is False   # :11-17
    m = P.QuantizedConv2d(16, 32, 3, 2, quantize_fn=P.PowerOfTwoQuantizer, bits=3)
    assert isinstance(m, torch.nn.Conv2d) and list(m.state_dict()) == ["weight"]
    assert m.quantize_fn is P.PowerOfTwoQuantizer and m.bits == 3
    g = torch.ones(3)
    assert P.PowerOfTwoQuantizer.backward(None, g)[0] is g and P.PowerOfTwoPlusQuantizer.backward(None, g)[1:] == (None, None)
    from drop_in.utils.quantizers import quantizer_dict as qd2
    from drop_in.models.quantized_conv import QuantizedConv2d as qc2
    assert qd2 is P.quantizer_dict and qc2 is P.QuantizedConv2d


def test_lin_quantizers_match_reference_vectors():
    z = G.load("lin_golden.npz")
    w = torch.from_numpy(z["w"])
    for name, cls in (("lin", P.LinearPowerOfTwoQuantizer), ("lin+", P.LinearPowerOfTwoPlusQuantizer)):
        for bits in (3, 4):
            got = cls.forward(None, w, bits=bits).numpy()
            assert np.array_equal(got.view(np.uint32), z[f"{name}|{bits}"].view(np.uint32)), (name, bits)


@pytest.fixture
def oracle_backend(monkeypatch):
    """Route the two quantizer ops through the oracle (TEST fake backend, never shipped)."""
    from oracle.po2_oracle_torch import quantize_ref

    def fake_quantize(x, bits, fsr, plus):
        return quantize_ref(x.detach(), bits, fsr, plus)

    def fake_full(x, bits, fsr, plus):
        y = quantize_ref(x.detach(), bits, fsr, plus)
        return (y, torch.zeros(1, dtype=torch.uint8), x.detach().abs().max().float(),
                torch.zeros((), dtype=torch.int32), ((y - x.detach()).double() ** 2).sum())
    monkeypatch.setattr(ops, "quantize", fake_quantize)
    monkeypatch.setattr(ops, "quantize_full", fake_full)
    monkeypatch.setattr(ops, "_require_cuda", lambda t, what: None)
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True), raising=False)
    yield
    

def test_quantize_model_control_flow_and_known_answers(oracle_backend):
    """utils/quantizers.py:139-153 on the seeded ResNet-20: the reference's own MSE values."""
    from workloads import resnet_cifar
    ka = G.load("known_answers.npz")
    for qn, Q in (("po2", P.PowerOfTwoQuantizer), ("po2+", P.PowerOfTwoPlusQuantizer)):
        for bits in (3, 4):
            torch.manual_seed(8)
            model = resnet_cifar(20, 10, None, bits)
            before = copy.deepcopy(model.state_dict())
            mse = P.quantize_model(model, Q, bits)
            assert abs(mse - float(ka[f"resnet20_ptq_mse|{qn}|{bits}"])) <= 2e-6 * mse
            after = model.state_dict()
            changed = [k for k in before if not torch.equal(before[k], after[k])]
            qconv = [n + ".weight" for n, m in model.named_modules() if isinstance(m, P.QuantizedConv2d)]
            assert sorted(changed) == sorted(qconv) and len(qconv) == 20       # stem conv / fc untouched
            assert "conv1.weight" not in changed
            assert all(hasattr(m, "_po2_ptq") for m in model.modules() if isinstance(m, P.QuantizedConv2d))


def test_quantize_model_without_quantized_layers_raises():
    with pytest.raises(ZeroDivisionError):
        P.quantize_model(torch.nn.Sequential(torch.nn.Conv2d(3, 3, 1)), P.PowerOfTwoQuantizer, 4)


def test_flavor_and_mode_switches():
    assert P.get_log2_flavor() in ("ieee", "torch_cuda")
    with pytest.raises(ValueError):
        P.set_log2_flavor("glibc")
    with pytest.raises(ValueError):
        ops.set_conv_mode("magic")
    P.set_log2_flavor("torch_cuda")
    assert P.get_log2_flavor() == "torch_cuda"
    P.set_log2_flavor("ieee")


def test_fused_sync_batchnorm_cpu_fallback_and_state_dict():
    """FusedSyncBatchNorm on CPU tensors takes nn.SyncBatchNorm's own path (+ add, + activation): same
    numbers as the stock modules, same state_dict keys, every activation variant."""
    import torch.nn as nn
    import torch.nn.functional as F
    torch.manual_seed(0)
    x = torch.randn(6, 8, 5, 5)
    res = torch.randn(6, 8, 5, 5)
    for act, fn in ((None, lambda t: t), ("relu", F.relu), ("relu6", F.relu6), ("silu", F.silu)):
        mine = P.FusedSyncBatchNorm(8, act=act)
        stock = nn.BatchNorm2d(8)
        assert list(mine.state_dict()) == list(stock.state_dict())
        mine.load_state_dict(stock.state_dict())
        for train in (True, False):
            mine.train(train), stock.train(train)
            assert torch.allclose(mine(x), fn(stock(x)), atol=1e-6), (act, train)
        assert torch.allclose(mine(x, res), fn(stock(x) + res), atol=1e-6)
    m = P.FusedSyncBatchNorm(8)
    assert torch.allclose(m(x, res, True), F.relu(nn.BatchNorm2d(8)(x) + res), atol=1e-6)   # per-call relu=True
    with pytest.raises(ValueError):
        P.FusedSyncBatchNorm(8, act="gelu")


def test_workloads_keep_state_dict_keys_with_fused_norms():
    """The fused-norm variants of the three model families have exactly the stock variants' state_dict
    keys and shapes (an nn.Identity keeps the nn.Sequential indices where an activation module was)."""
    from workloads import mobilenet_v2_cifar, mobilevit_xs, resnet_cifar
    import torch.nn as nn
    pairs = [(resnet_cifar(20, 10, None, 4), resnet_cifar(20, 10, None, 4, norm_cls=nn.SyncBatchNorm)),
             (mobilenet_v2_cifar(10, None, 4, fused_norm=True), mobilenet_v2_cifar(10, None, 4, fused_norm=False)),
             (mobilevit_xs((32, 32), 10, (1, 1), None, 8, fused_norm=True), mobilevit_xs((32, 32), 10, (1, 1), None, 8, fused_norm=False))]
    for a, b in pairs:
        sa, sb = a.state_dict(), b.state_dict()
        assert list(sa) == list(sb)
        assert all(sa[k].shape == sb[k].shape for k in sa)
        assert any(isinstance(m, P.FusedSyncBatchNorm) for m in a.modules())
        assert not any(isinstance(m, P.FusedSyncBatchNorm) for m in b.modules())


def test_conv_shape_validation_raises_like_nn_conv2d():
    """ops.check_conv_shapes: the RuntimeErrors nn.Conv2d / the reference raise for a wrong channel count,
    indivisible groups or a kernel larger than the padded input (ADVICE r1: the C ABI has no
    weight-channel argument, so the host must catch these before any launch)."""
    from po2_quantization_b200 import ops
    ops.check_conv_shapes((2, 16, 8, 8), (32, 16, 3, 3), 1, 1)
    ops.check_conv_shapes((2, 16, 8, 8), (16, 1, 3, 3), 16, 1)
    with pytest.raises(RuntimeError, match="expected input.* to have 16 channels, but got 24"):
        ops.check_conv_shapes((2, 24, 8, 8), (32, 16, 3, 3), 1, 1)
    with pytest.raises(RuntimeError, match="divisible"):
        ops.check_conv_shapes((2, 16, 8, 8), (30, 4, 3, 3), 4, 1)
    with pytest.raises(RuntimeError, match="Kernel size"):
        ops.check_conv_shapes((2, 16, 1, 1), (32, 16, 3, 3), 1, 0)
    with pytest.raises(RuntimeError, match="4D"):
        ops.check_conv_shapes((16, 8, 8), (32, 16, 3, 3), 1, 1)
    # the same errors as torch's own convolution
    conv = torch.nn.Conv2d(16, 32, 3, padding=1, bias=False)
    with pytest.raises(RuntimeError, match="to have 16 channels, but got 24"):
        conv(torch.randn(2, 24, 8, 8))


def test_library_paths_are_reported_and_strict_mode_raises(monkeypatch):
    from po2_quantization_b200 import _lib, ops
    ops._noted.discard("t:why")
    with pytest.warns(RuntimeWarning, match="because"):
        ops.note_library_path("t:why", "because")
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        ops.note_library_path("t:why", "because")            # second time: silent
    monkeypatch.setenv("PO2_STRICT", "1")
    with pytest.raises(_lib.Po2Error, match="because"):
        ops.note_library_path("t:why", "because")


def test_batch_sharded_rejects_a_second_backward_before_averaging():
    """ADVICE r1: with overlap=True a bucket is reduced from the grad hooks; a second backward() before
    average_gradients() must raise instead of silently mixing averaged and local gradients."""
    from po2_quantization_b200.distributed import BatchSharded
    m = BatchSharded(torch.nn.Linear(4, 2))
    m._buckets = [list(m.module.parameters())]
    m._bucket_of = {id(p): 0 for p in m._buckets[0]}
    m._pending = [-1]                                         # state after the bucket's all-reduce was launched
    with pytest.raises(RuntimeError, match="average_gradients"):
        m._on_grad(m._buckets[0][0])


def test_reference_file_loader_variants():
    """workloads/reference_files.py: the reference's model files import on the drop-in shims and on
    their own classes, side by side, without leaking `models` / `utils` into sys.modules."""
    import sys
    from workloads import reference_files as RF
    if RF.find_reference() is None:
        pytest.skip("no reference checkout ($PO2_REFERENCE or baseline/_ref)")
    d, s = RF.load("dropin"), RF.load("stock")
    assert d.QuantizedConv2d is P.QuantizedConv2d and s.QuantizedConv2d is not P.QuantizedConv2d
    assert d.quantizers.quantizer_dict["po2+"] is P.PowerOfTwoPlusQuantizer
    assert not any(k == "models" or k.startswith("models.") for k in sys.modules)
    torch.manual_seed(8)
    a = s.get_model("resnet20", 10, None, 4, (32, 32))
    b = d.get_model("resnet20", 10, None, 4, (32, 32))
    b.load_state_dict(a.state_dict(), strict=True)
    x = torch.randn(2, 3, 32, 32)
    a.eval(); b.eval()
    with torch.no_grad():
        assert torch.equal(a(x), b(x))
    v = RF.mobilevit_224(s)
    assert sum(1 for m in v.modules() if isinstance(m, s.QuantizedConv2d)) == 33


def test_fuse_batchnorm_and_fold_conv_bn_rewrite_the_module_tree():
    """fold.py on CPU: fuse_batchnorm re-classes nn.SyncBatchNorm instances in place (same state_dict keys) and moves
    an activation behind a norm in an nn.Sequential into the norm; fold_conv_bn pairs conv + norm for inference; the
    functional conv_bn_act falls back to the separate calls for CPU tensors and gives the same numbers."""
    import torch.nn as nn
    import torch.nn.functional as F
    seq = nn.Sequential(P.QuantizedConv2d(4, 8, 3), nn.SyncBatchNorm(8), nn.ReLU6(inplace=True),
                        P.QuantizedConv2d(8, 8, 1, padding=0), nn.SyncBatchNorm(8))
    keys = list(seq.state_dict().keys())
    assert P.fuse_batchnorm(seq) == 2
    assert list(seq.state_dict().keys()) == keys
    assert type(seq[1]) is P.FusedSyncBatchNorm and seq[1].act == "relu6" and isinstance(seq[2], nn.Identity)
    assert type(seq[4]) is P.FusedSyncBatchNorm and seq[4].act is None
    seq.eval()
    with torch.no_grad():
        seq[1].running_mean.normal_(); seq[1].running_var.uniform_(0.5, 2.0)
        x = torch.randn(2, 4, 6, 6)
        ref = seq(x)
        assert P.fold_conv_bn(seq) == 2
        assert isinstance(seq[0], P.FoldedConvBN) and isinstance(seq[1], nn.Identity)
        assert torch.allclose(seq(x), ref, atol=1e-6)
        # functional form, CPU tensors: conv, norm, add, ReLU as separate torch ops
        conv, bn = P.QuantizedConv2d(4, 4, 3), P.FusedSyncBatchNorm(4).eval()
        r = torch.randn(2, 4, 6, 6)
        out = P.conv_bn_act(conv, bn, x, r, True)
        assert torch.allclose(out, F.relu(bn(conv(x)) + r), atol=1e-6)


def test_argument_errors_and_planning_queries_of_the_round_2_entry_points_abi_v2():
    import ctypes
    from po2_quantization_b200 import _lib
    lib = _lib.load()
    one = ctypes.c_void_p(4096)
    conv = (8, 16, 32, 32, 16, 3, 3)
    # planning queries answer on the host (no GPU): kernel kinds, pack sizes
    assert lib.po2_conv2d_kernel_kind(128, 960, 1, 1, 320, 1, 1, 1, 0, 1, 2) == 4          # small-map pointwise GEMM
    assert lib.po2_conv2d_kernel_kind(128, 96, 16, 16, 96, 3, 3, 2, 1, 96, 2) == 1          # depthwise
    assert lib.po2_conv2d_kernel_kind(*conv, 2, 1, 1, 2) == 2                               # stride 2: register-fed tcgen05
    assert lib.po2_conv2d_kernel_kind(*conv, 1, 1, 1, 1) == 0                               # fp32 mode: direct
    assert lib.po2_conv2d_wgrad_kernel_kind(*conv, 2, 1, 1, 2) == 0                          # stride 2 goes through po2_dilate2
    assert lib.po2_conv2d_pack_bytes(128, 960, 1, 1, 320, 1, 1, 1, 0, 1, 2) == 0             # no packed operand for kind 4
    assert lib.po2_conv2d_depthwise_wgrad_workspace(96) > 4096 * 4
    # argument errors come back as PO2_E_* before any launch
    assert lib.po2_conv2d_fwd_ep(one, one, one, one, *conv, 1, 1, 1, 0, 4, 1, 2, one, 1 << 20, one, one, None, 7, None) == -9
    assert lib.po2_conv2d_fwd_ep(one, one, one, one, *conv, 1, 1, 1, 0, 4, 1, 2, one, 1 << 20, one, None, None, 0, None) == -3
    assert lib.po2_conv2d_fwd_packed_ep(one, one, one, one, *conv, 1, 1, 1, 2, None, None, one, 0, None) == -3   # residual without affine
    assert lib.po2_dilate2(one, one, 4, 8, 7, None) == -10                                    # odd width
    assert lib.po2_dilate2(None, one, 4, 8, 8, None) == -3
    assert lib.po2_conv2d_depthwise_dgrad(one, None, one, 2, 8, 4, 4, None) == -3
    assert lib.po2_conv2d_depthwise_wgrad(one, one, one, 2, 8, 4, 4, one, 16, None) == -8
    assert lib.po2_bn_bwd_fused(one, None, one, one, one, one, one, one, None, None, one, None, 4, 8, 16, 64, one, 1 << 20, None) == -9
    assert lib.po2_bn_bwd_fused(one, one, one, None, one, one, one, one, None, None, one, one, 3, 8, 16, 64, one, 1 << 20, None) == -9
    assert lib.po2_conv2d_dgrad_packed(one, None, one, one, *conv, 1, 2, None) == -3
    # the multi-tensor SGD step: host arrays of device pointers, checked before the launch
    ptrs = (ctypes.c_void_p * 2)(4096, 8192)
    odd = (ctypes.c_void_p * 2)(4096, 8193)
    n2 = (ctypes.c_longlong * 2)(16, 5)
    assert lib.po2_sgd_max_tensors_per_launch() == 96
    assert lib.po2_sgd_step(ptrs, ptrs, ptrs, n2, 0, 0.1, 0.9, 1e-4, 0, None) == 0                  # nothing to do
    assert lib.po2_sgd_step(ptrs, ptrs, ptrs, n2, -1, 0.1, 0.9, 1e-4, 0, None) == -4
    assert lib.po2_sgd_step(ptrs, ptrs, None, n2, 2, 0.1, 0.9, 1e-4, 0, None) == -3                 # momentum needs buffers
    assert lib.po2_sgd_step(ptrs, odd, ptrs, n2, 2, 0.1, 0.9, 1e-4, 0, None) == -5                  # not a float address
    assert lib.po2_sgd_step(ptrs, ptrs, ptrs, (ctypes.c_longlong * 2)(16, 0), 2, 0.1, 0.9, 1e-4, 0, None) == -4


def test_sgd_subclass_delegates_what_the_kernel_does_not_take():
    """optim.SGD on CPU parameters (and Nesterov / dampening groups anywhere) is torch.optim.SGD's own step: same
    numbers, same state layout, interchangeable state_dict -- the kernel path is CUDA fp32 only and is covered by
    tests/test_models_gpu.py."""
    torch.manual_seed(0)
    a = [torch.nn.Parameter(torch.randn(5, 3)), torch.nn.Parameter(torch.randn(7))]
    b = [torch.nn.Parameter(p.detach().clone()) for p in a]
    oa = P.optim.SGD(a, lr=0.1, momentum=0.9, weight_decay=1e-4)
    ob = torch.optim.SGD(b, lr=0.1, momentum=0.9, weight_decay=1e-4)
    assert isinstance(oa, torch.optim.SGD)
    for step in range(3):
        for pa, pb in zip(a, b):
            g = torch.randn(pa.shape)
            pa.grad, pb.grad = g.clone(), g.clone()
        assert oa.step(lambda: torch.tensor(1.5)).item() == 1.5          # the closure protocol
        ob.step()
    for pa, pb in zip(a, b):
        assert torch.equal(pa, pb)
        assert torch.equal(oa.state[pa]["momentum_buffer"], ob.state[pb]["momentum_buffer"])
    ob.load_state_dict(oa.state_dict())
    # a parameter without a gradient is skipped, like in torch
    a[1].grad = None
    before = a[1].detach().clone()
    a[0].grad = torch.ones_like(a[0])
    oa.step()
    assert torch.equal(a[1], before)


def test_round_2_switches_and_planning_queries_on_the_host_abi_v2():
    import ctypes
    from po2_quantization_b200 import _lib, batchnorm
    lib = _lib.load()
    one = ctypes.c_void_p(4096)
    # weight gradients on a side stream: a process-wide switch, off unless asked for
    was = ops.get_wgrad_overlap()
    try:
        ops.set_wgrad_overlap(True)
        assert ops.get_wgrad_overlap() is True
        ops.join_weight_gradients()                         # nothing pending: a no-op, also without a GPU
    finally:
        ops.set_wgrad_overlap(was)
    # the skip-connection routing only applies to tensors produced by the fused norm's autograd node
    t = torch.randn(2, 3, requires_grad=True) * 2
    assert batchnorm._route_skip_gradient(t) is t
    # the stem's weight-gradient kernel: which shapes it takes is a host-side question
    assert lib.po2_conv2d_stem_wgrad_workspace(128, 3, 64, 64, 24, 3, 3, 1, 1, 1) == 0               # g[n] does not fit shared memory
    assert lib.po2_conv2d_stem_wgrad_workspace(128, 16, 32, 32, 16, 3, 3, 1, 1, 1) == 0              # not a small-C layer
    assert lib.po2_conv2d_stem_wgrad_workspace(128, 3, 32, 32, 16, 3, 3, 2, 1, 1) == 0               # stride 2
    assert lib.po2_conv2d_stem_wgrad(one, one, one, 128, 3, 32, 32, 16, 3, 3, 1, 1, 1, None, 0, None) == -3
    assert lib.po2_conv2d_stem_wgrad(one, one, one, 128, 3, 32, 32, 16, 5, 5, 1, 2, 1, one, 1 << 20, None) == -10
    m = torch.nn.Sequential(torch.nn.Conv2d(3, 16, 3, 1, 1, bias=False), torch.nn.Conv2d(16, 16, 3, 1, 1, bias=False),
                            torch.nn.Conv2d(3, 8, 3, 2, 1, bias=False), torch.nn.Conv2d(3, 8, 3, 1, 1, bias=True))
    keys = list(m.state_dict())
    assert P.accelerate_stem(m) == 1 and isinstance(m[0], P.StemConv2d) and type(m[1]) is torch.nn.Conv2d
    assert list(m.state_dict()) == keys
    assert m[0](torch.randn(2, 3, 8, 8)).shape == (2, 16, 8, 8)                                     # CPU: nn.Conv2d's own forward
