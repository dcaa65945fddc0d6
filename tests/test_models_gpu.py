"""Model-level GPU parity: (1) QAT convergence of the operand modes against the reference's own
arithmetic over 50 optimizer steps, (2) the reference's OWN model files (baseline/_ref, staged from the
unmodified checkout) running on the drop-in classes on the B200 against the same files on their stock
torch path, (3) the argument errors nn.Conv2d raises.  Results that are worth keeping are also written
to gpurun_out/ (copied to profiles/ by hand)."""
import json
import os

import pytest
import torch
import torch.nn as nn

pytestmark = pytest.mark.gpu

import po2_quantization_b200 as P  # noqa: E402
from po2_quantization_b200 import ops  # noqa: E402

OUT = os.path.join(os.environ.get("GRAFT_REPO_ROOT", os.path.dirname(os.path.dirname(os.path.abspath(__file__)))), "gpurun_out")


def _dump(name, obj):
    try:
        os.makedirs(OUT, exist_ok=True)
        json.dump(obj, open(os.path.join(OUT, name), "w"), indent=1)
    except OSError:
        pass


def _learnable_batches(n_batches=4, batch=64, seed=0):
    """a small fixed data set whose labels are a function of the images, so that the loss really falls"""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n_batches * batch, 3, 32, 32, generator=g)
    proj = torch.randn(10, 3 * 8 * 8, generator=g)
    y = (torch.nn.functional.avg_pool2d(x, 4).flatten(1) @ proj.t()).argmax(1)
    return [(x[i * batch:(i + 1) * batch], y[i * batch:(i + 1) * batch]) for i in range(n_batches)]


def _train_curve(model, batches, steps, lr=0.05):
    opt = torch.optim.SGD(model.parameters(), lr=lr, momentum=0.9, weight_decay=1e-4)
    crit = nn.CrossEntropyLoss()
    losses = []
    for i in range(steps):
        x, y = batches[i % len(batches)]
        opt.zero_grad()
        loss = crit(model(x), y)
        loss.backward()
        opt.step()
        losses.append(loss.detach())
    return [float(v) for v in torch.stack(losses).cpu()]


def _smooth(c, k=8):
    return [sum(c[max(0, i - k + 1):i + 1]) / len(c[max(0, i - k + 1):i + 1]) for i in range(len(c))]


def test_qat_loss_curves_bf16_tf32_fp32_track_the_reference():
    """50 SGD steps of ResNet-20 PO2 4-bit QAT (train-mode BatchNorm, momentum 0.9) from identical
    weights on identical data: the bf16-operand mode (default), the tf32-operand mode and the
    fp32-accumulate mode of this library against the reference's arithmetic on the same GPU in true fp32
    (stock ATen quantizer ops + cuDNN with allow_tf32=False) and in the reference's own default (cuDNN
    TF32).  Training is chaotic, so curves are compared after smoothing: every mode must stay within a
    band of the fp32 reference no wider than twice the band the reference's OWN TF32 default shows, and
    must reach the same final loss level."""
    from oracle.po2_oracle_torch import PO2, QuantizedConv2dOracle
    from workloads import resnet_cifar
    steps = 50
    batches = [(x.cuda(), y.cuda()) for x, y in _learnable_batches()]
    torch.manual_seed(8)
    init = resnet_cifar(20, 10, PO2, 4, conv_cls=QuantizedConv2dOracle).state_dict()
    curves = {}
    old_tf32 = torch.backends.cudnn.allow_tf32
    try:
        for name, tf32 in (("reference_fp32", False), ("reference_tf32_default", True)):
            torch.backends.cudnn.allow_tf32 = tf32
            m = resnet_cifar(20, 10, PO2, 4, conv_cls=QuantizedConv2dOracle)
            m.load_state_dict(init)
            curves[name] = _train_curve(m.cuda().train(), batches, steps)
        torch.backends.cudnn.allow_tf32 = False          # the stem conv of our models stays true fp32
        for name, mode in (("po2_bf16_operands", "tc"), ("po2_tf32_operands", "tf32"), ("po2_fp32_accumulate", "fp32")):
            ops.set_conv_mode(mode)
            m = resnet_cifar(20, 10, P.PowerOfTwoQuantizer, 4)
            m.load_state_dict(init)
            curves[name] = _train_curve(m.cuda().train(), batches, steps)
    finally:
        torch.backends.cudnn.allow_tf32 = old_tf32
        ops.set_conv_mode(ops.DEFAULT_CONV_MODE)
    ref = _smooth(curves["reference_fp32"])
    band = {k: max(abs(a - b) for a, b in zip(_smooth(v), ref)) for k, v in curves.items()}
    final = {k: sum(v[-10:]) / 10 for k, v in curves.items()}
    _dump("qat_loss_curves_resnet20.json", {"steps": steps, "curves": curves, "max_smoothed_gap_vs_reference_fp32": band,
                                            "mean_loss_last_10_steps": final})
    assert final["reference_fp32"] < 0.8 * curves["reference_fp32"][0], "the reference itself did not learn"
    allowed = max(2.0 * band["reference_tf32_default"], 0.08 * curves["reference_fp32"][0])
    for k in ("po2_bf16_operands", "po2_tf32_operands", "po2_fp32_accumulate"):
        assert band[k] <= allowed, (k, band[k], allowed, band)
        assert abs(final[k] - final["reference_fp32"]) <= 0.15 * curves["reference_fp32"][0], (k, final)
        assert final[k] < 0.8 * curves[k][0], (k, "did not learn", final[k], curves[k][0])


# ------------------------------------------------------------------------------------------------
# the reference's own model files on the B200
# ------------------------------------------------------------------------------------------------
def _ref_ns():
    from workloads import reference_files as RF
    d, s = RF.load("dropin"), RF.load("stock")
    if d is None or s is None:
        pytest.skip("no reference checkout ($PO2_REFERENCE or baseline/_ref)")
    return RF, d, s


@pytest.mark.parametrize("name,bits", [("resnet20", 4), ("resnet56", 4), ("mobilenet", 4), ("mobilevit", 4)])
def test_reference_model_files_ptq_forward_on_gpu(name, bits):
    """models/{resnet,mobilenet,mobile_vit}.py UNMODIFIED: built once on the drop-in classes (our kernels)
    and once on the reference's own classes (stock torch), same weights; quantize_model + eval forward on
    the GPU.  Quantized weights bit-equal, MSE equal, logits within the bf16 tolerance, and -- in
    fp32-accumulate mode -- identical top-1 (north_star (c))."""
    RF, d, s = _ref_ns()
    torch.manual_seed(8)
    ref = s.get_model(name, 10, None, bits, (32, 32))
    mine = d.get_model(name, 10, None, bits, (32, 32))
    mine.load_state_dict(ref.state_dict(), strict=True)
    ref, mine = ref.cuda().eval(), mine.cuda().eval()
    nq = sum(1 for m in mine.modules() if isinstance(m, P.QuantizedConv2d))
    assert nq == {"resnet20": 20, "resnet56": 56, "mobilenet": 50, "mobilevit": 33}[name]
    mse_ref = s.quantizers.quantize_model(ref, s.quantizers.PowerOfTwoPlusQuantizer, bits)
    ops.set_log2_flavor("torch_cuda")                 # the reference ran on THIS GPU: compare under its log2 flavor
    try:
        mse = d.quantizers.quantize_model(mine, d.quantizers.PowerOfTwoPlusQuantizer, bits)
    finally:
        ops.set_log2_flavor("ieee")
    assert abs(mse - mse_ref) <= 1e-5 * mse_ref
    for (k, a), (_, b) in zip(mine.state_dict().items(), ref.state_dict().items()):
        assert torch.equal(a, b), f"{k}: PTQ weights differ from the reference's on this GPU"
    x = torch.randn(64, 3, 32, 32, generator=torch.Generator().manual_seed(0)).cuda()
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            ops.LAUNCHES = 0
            out = mine(x)
            assert ops.LAUNCHES >= nq, "the reference model file did not reach the po2 conv kernels"
            want = ref(x)
            rel = ((out.double() - want.double()).abs().max() / want.double().abs().max()).item()
            assert rel < 1e-2, (name, rel)
            ops.set_conv_mode("fp32")
            try:
                out32 = mine(x)
            finally:
                ops.set_conv_mode(ops.DEFAULT_CONV_MODE)
            rel32 = ((out32.double() - want.double()).abs().max() / want.double().abs().max()).item()
            assert rel32 < 1e-4, (name, rel32)
            assert torch.equal(out32.argmax(1), want.argmax(1)), "top-1 differs in fp32-accumulate mode"
    finally:
        torch.backends.cudnn.allow_tf32 = old
    err, numel = mine.get_quantization_error()        # quantize_fn=None after PTQ: (0, numel) per layer
    assert err == 0 and numel > 0


@pytest.mark.parametrize("name", ["resnet20", "mobilenet"])
def test_reference_model_files_qat_step_on_gpu(name):
    """One QAT training step (train.py:79-92) of the reference's own model file on the drop-in classes vs
    the same file on the reference's classes, fp32-accumulate mode: loss and every weight gradient."""
    RF, d, s = _ref_ns()
    torch.manual_seed(8)
    ref = s.get_model(name, 10, s.quantizers.PowerOfTwoQuantizer, 4, (32, 32))
    mine = d.get_model(name, 10, P.PowerOfTwoQuantizer, 4, (32, 32))
    mine.load_state_dict(ref.state_dict(), strict=True)
    train_bn = name == "resnet20"                      # see test_qat_training_step_matches_oracle_model
    ref, mine = ref.cuda().train(train_bn), mine.cuda().train(train_bn)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(32, 3, 32, 32, generator=g).cuda()
    y = torch.randint(0, 10, (32,), generator=g).cuda()
    crit = nn.CrossEntropyLoss()
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    ops.set_conv_mode("fp32")
    ops.set_log2_flavor("torch_cuda")
    try:
        lr_ = crit(ref(x), y); lr_.backward()
        lm = crit(mine(x), y); lm.backward()
    finally:
        ops.set_conv_mode(ops.DEFAULT_CONV_MODE)
        ops.set_log2_flavor("ieee")
        torch.backends.cudnn.allow_tf32 = old
    assert abs(lm.item() - lr_.item()) < 5e-3 * max(1.0, abs(lr_.item()))
    pr = dict(ref.named_parameters())
    gscale = max(v.grad.double().pow(2).mean().sqrt().item() for v in pr.values())
    checked = 0
    for k, p in mine.named_parameters():
        assert p.grad is not None, k
        gr = pr[k].grad.double()
        if gr.pow(2).mean().sqrt().item() < 1e-7 * gscale or p.numel() < 64:
            continue
        rel = ((p.grad.double() - gr).pow(2).mean().sqrt() / gr.pow(2).mean().sqrt()).item()
        assert rel < 3e-2, (k, rel)
        checked += 1
    assert checked >= 10
    # the model-level error walker (train.py:106) on the drop-in classes == on the reference's
    e1, n1 = mine.get_quantization_error()
    e2, n2 = ref.get_quantization_error()
    assert n1 == n2 and abs(float(e1) - float(e2)) <= 1e-5 * float(e2)


def test_conv_argument_errors_match_nn_conv2d():
    """A wrong channel count must raise like nn.Conv2d / the reference do (RuntimeError), never read out
    of bounds: module forward (QAT, PTQ, prefetched), the ops, and the raw launchers."""
    conv = P.QuantizedConv2d(16, 32, 3, quantize_fn=P.PowerOfTwoQuantizer, bits=4).cuda()
    good, bad = torch.randn(2, 16, 8, 8, device="cuda"), torch.randn(2, 24, 8, 8, device="cuda")
    conv(good)
    with pytest.raises(RuntimeError, match="channels"):
        conv(bad)
    seq = nn.Sequential(P.QuantizedConv2d(16, 32, 3)).cuda()
    P.quantize_model(seq, P.PowerOfTwoQuantizer, 4)
    with torch.no_grad():
        seq(good)
        with pytest.raises(RuntimeError, match="channels"):
            seq(bad)
    w = torch.randn(32, 16, 3, 3, device="cuda")
    qw, scale = torch.ops.po2.quantize_scaled(w, 4, 1, False)
    with pytest.raises(RuntimeError, match="channels"):
        torch.ops.po2.conv2d(bad, qw, scale, 1, 1, 1, 0)
    with pytest.raises(RuntimeError, match="channels"):
        torch.ops.po2.qconv2d(bad, w, 4, 1, False, 1, 1, 1, 0)
    packed = ops.conv2d_pack(qw, scale, tuple(good.shape), 1, 1, 1, 0)
    torch.ops.po2.conv2d_packed(good, packed, scale, 32, 3, 3, 1, 1, 1, 0)
    with pytest.raises(RuntimeError, match="packed operand"):
        torch.ops.po2.conv2d_packed(bad, packed, scale, 32, 3, 3, 1, 1, 1, 0)
    with pytest.raises(RuntimeError, match="Kernel size"):
        torch.ops.po2.conv2d(torch.randn(1, 16, 1, 1, device="cuda"), qw, scale, 1, 0, 1, 0)


def test_library_fallbacks_are_loud(monkeypatch):
    """configurations the kernels do not take run nn.Conv2d's own path WITH a warning (once per reason),
    and raise under PO2_STRICT=1"""
    conv = P.QuantizedConv2d(8, 8, 3, dilation=2, padding=2, quantize_fn=P.PowerOfTwoQuantizer, bits=4).cuda()
    x = torch.randn(1, 8, 8, 8, device="cuda")
    ops._noted.clear()
    with pytest.warns(RuntimeWarning, match="dilation"):
        conv(x)
    monkeypatch.setenv("PO2_STRICT", "1")
    with pytest.raises(P._lib.Po2Error, match="dilation"):
        conv(x)


# ------------------------------------------------------------------------------------------------
# SURVEY.md section 8f row 4: fused error sums for all layers, packed-code checkpoints
# ------------------------------------------------------------------------------------------------
def test_quantization_error_comes_from_the_quantizer_pass():
    """QuantizedConv2d.get_quantization_error (models/quantized_conv.py:40-45) and the model-level sum
    (models/resnet.py:214-224, train.py:106): equal to sum((Q(w)-w)^2) from the numpy oracle to 1e-6, one
    launch per layer without the prefetch and NO launch at all once the multi-tensor prefetch has run."""
    import numpy as np
    from oracle import po2_oracle as O
    from workloads import resnet_cifar
    torch.manual_seed(8)
    model = resnet_cifar(20, 10, P.PowerOfTwoPlusQuantizer, 4).cuda().train()
    convs = [m for m in model.modules() if isinstance(m, P.QuantizedConv2d)]
    want = []
    for m in convs:
        w = m.weight.detach().cpu().numpy().ravel()
        want.append(float(np.sum((O.po2_plus(w, 4).astype(np.float64) - w.astype(np.float64)) ** 2)))
    ops.LAUNCHES = 0
    got = [m.get_quantization_error() for m in convs]
    assert ops.LAUNCHES == len(convs)                       # one fused launch each (the reference: 12 ATen launches each)
    for (e, n), w_, m in zip(got, want, convs):
        assert n == m.weight.numel() and abs(e.item() - w_) <= 1e-6 * w_, (e.item(), w_)
    P.enable_weight_prefetch(model)
    x = torch.randn(8, 3, 32, 32, device="cuda")
    model(x); model(x)                                       # first forward records the shapes, second prefetches
    ops.LAUNCHES = 0
    tot, numel = P.model_quantization_error(model)
    assert ops.LAUNCHES == 0, "the prefetched error sums were not used"
    assert numel == sum(m.weight.numel() for m in convs)
    assert abs(tot.item() - sum(want)) <= 1e-6 * sum(want)
    # a weight update invalidates the cached value
    with torch.no_grad():
        convs[3].weight.mul_(1.5)
    w = convs[3].weight.detach().cpu().numpy().ravel()
    e, _ = convs[3].get_quantization_error()
    ref = float(np.sum((O.po2_plus(w, 4).astype(np.float64) - w.astype(np.float64)) ** 2))
    assert abs(e.item() - ref) <= 1e-6 * ref


@pytest.mark.parametrize("bits,plus", [(4, True), (4, False), (8, True), (3, False)])
def test_packed_checkpoint_round_trip_is_bit_exact(tmp_path, bits, plus):
    """state_dict -> packed codes + scales -> state_dict: bit-identical for a PTQ model (exact zeros and
    the DDP 'module.' prefix included); for a QAT model the unpacked weights are exactly Q(w)."""
    from workloads import resnet_cifar
    Q = P.PowerOfTwoPlusQuantizer if plus else P.PowerOfTwoQuantizer
    torch.manual_seed(8)
    model = resnet_cifar(20, 10, None, bits).cuda()
    convs = [m for m in model.modules() if isinstance(m, P.QuantizedConv2d)]
    with torch.no_grad():
        convs[2].weight.view(-1)[::7] = 0.0                  # exact zeros have no code: they travel as a bitmask
    P.quantize_model(model, Q, bits)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    path = str(tmp_path / "ptq.po2")
    meta = P.save_packed_checkpoint(model, path)
    assert meta["raw_fallbacks"] == []
    ratio = meta["quantized_packed_bytes"] / meta["quantized_fp32_bytes"]
    assert ratio < (0.14 if bits <= 4 else 0.27), ratio
    back = P.load_packed_checkpoint(path)
    assert list(back) == list(sd)
    for k in sd:
        assert back[k].dtype == sd[k].dtype and torch.equal(back[k].cpu(), sd[k].cpu()), k
        if sd[k].dtype == torch.float32:
            assert torch.equal(back[k].view(torch.int32).cpu(), sd[k].view(torch.int32).cpu()), k
    fresh = resnet_cifar(20, 10, None, bits).cuda()
    fresh.load_state_dict(back, strict=True)
    # QAT model: master weights are NOT on the grid; the packed file holds what the forward convolves with
    torch.manual_seed(9)
    qat = resnet_cifar(20, 10, Q, bits).cuda()
    packed = P.pack_state_dict(qat)
    un = P.unpack_state_dict(packed)
    for name, m in qat.named_modules():
        if isinstance(m, P.QuantizedConv2d):
            assert torch.equal(un[name + ".weight"], Q.forward(None, m.weight.detach(), bits=bits)), name
    # DDP-style prefix survives
    wrapped = torch.nn.Sequential()
    wrapped.add_module("module", model)
    back2 = P.unpack_state_dict(P.pack_state_dict(wrapped))
    assert all(k.startswith("module.") for k in back2) and len(back2) == len(sd)
    for k in sd:
        assert torch.equal(back2["module." + k].cpu(), sd[k].cpu())


@pytest.mark.parametrize("family", ["resnet20", "mobilenet", "mobilevit"])
def test_folded_batchnorm_inference_matches_separate_kernels(family, monkeypatch):
    """PTQ inference with the eval-mode norms (+ residual add, + activation) folded into the conv epilogues
    (po2_quantization_b200/fold.py) against the same model running conv and norm as separate kernels: same
    logits up to fp32 rounding of the affine, same top-1; and far fewer launches."""
    import po2_quantization_b200 as P
    from po2_quantization_b200 import ops
    from workloads.mobilenet_cifar import mobilenet_v2_cifar
    from workloads.mobilevit import mobilevit_xs
    from workloads.resnet_cifar import resnet_cifar
    torch.manual_seed(3)
    if family == "resnet20":
        m, x = resnet_cifar(20, 10, None, 4), torch.randn(64, 3, 32, 32, device="cuda")
    elif family == "mobilenet":
        m, x = mobilenet_v2_cifar(10, None, 4), torch.randn(64, 3, 32, 32, device="cuda")
    else:
        m, x = mobilevit_xs((64, 64), 10, (2, 2), None, 8), torch.randn(8, 3, 64, 64, device="cuda")
    m = m.cuda()
    with torch.no_grad():                                   # non-trivial running statistics and affine parameters
        for mod in m.modules():
            if isinstance(mod, torch.nn.modules.batchnorm._BatchNorm):
                mod.running_mean.normal_(0, 0.2); mod.running_var.uniform_(0.5, 1.5)
                mod.weight.uniform_(0.7, 1.3); mod.bias.normal_(0, 0.1)
    P.quantize_model(m, P.PowerOfTwoPlusQuantizer, 8 if family == "mobilevit" else 4)
    m.eval()
    with torch.no_grad():
        monkeypatch.setenv("PO2_FOLD_BN", "0")
        ref = m(x)
        n0 = ops.LAUNCHES
        m(x)
        separate = ops.LAUNCHES - n0
        monkeypatch.setenv("PO2_FOLD_BN", "1")
        folded_pairs = P.fold_conv_bn(m)
        out = m(x)
        n0 = ops.LAUNCHES
        m(x)
        folded = ops.LAUNCHES - n0
    assert family == "resnet20" or folded_pairs > 0
    assert folded < separate, (folded, separate)
    rel = ((out - ref).abs().max() / ref.abs().max()).item()
    assert rel < 2e-4, rel
    margin = ref.topk(2, dim=1).values
    decisive = (margin[:, 0] - margin[:, 1]) > 1e-3 * ref.abs().max()
    assert torch.equal(out.argmax(1)[decisive], ref.argmax(1)[decisive])


def test_fuse_batchnorm_on_the_reference_model_files():
    """The reference's own models/resnet.py + ONE line (fuse_batchnorm): same state_dict keys, same training step
    (loss and gradients against the unconverted model, whose norms are torch's), norms on this library's kernels."""
    import copy
    import po2_quantization_b200 as P
    from po2_quantization_b200 import ops
    from workloads import reference_files as RF
    ns = RF.load("dropin")
    if ns is None:
        pytest.skip("no reference checkout ($PO2_REFERENCE or baseline/_ref)")
    torch.manual_seed(5)
    a = ns.get_model("resnet20", 10, P.PowerOfTwoQuantizer, 4, (32, 32)).cuda().train()
    b = copy.deepcopy(a)
    keys = list(b.state_dict().keys())
    n = P.fuse_batchnorm(b)
    assert n == 19 + 2 and list(b.state_dict().keys()) == keys
    assert all(type(m) is P.FusedSyncBatchNorm for m in b.modules() if isinstance(m, torch.nn.SyncBatchNorm))
    x = torch.randn(32, 3, 32, 32, device="cuda")
    yl = torch.randint(0, 10, (32,), device="cuda")
    la = torch.nn.functional.cross_entropy(a(x), yl); la.backward()
    n0 = ops.LAUNCHES
    lb = torch.nn.functional.cross_entropy(b(x), yl); lb.backward()
    assert ops.LAUNCHES - n0 > 19 * 4                      # convs AND norms launched from libpo2b200.so
    assert abs(la.item() - lb.item()) < 1e-3 * abs(la.item())
    for (ka, pa), (kb, pb) in zip(a.named_parameters(), b.named_parameters()):
        assert ka == kb
        cos = torch.nn.functional.cosine_similarity(pa.grad.flatten(), pb.grad.flatten(), dim=0).item()
        assert cos > 0.98, (ka, cos)
    for (ka, ba), (kb, bb) in zip(a.named_buffers(), b.named_buffers()):
        assert torch.allclose(ba.float(), bb.float(), rtol=1e-4, atol=1e-5), ka
    # MobileNetV2 / MobileViT: the activation behind a norm inside an nn.Sequential moves into the norm
    m = ns.get_model("mobilenet", 10, P.PowerOfTwoPlusQuantizer, 4, (32, 32)).cuda()
    P.fuse_batchnorm(m)
    assert sum(1 for mod in m.modules() if isinstance(mod, P.FusedSyncBatchNorm) and mod.act == "relu6") >= 30
    assert not any(isinstance(mod, torch.nn.ReLU6) for mod in m.modules())


def test_weight_gradients_on_the_side_stream_are_the_same_gradients():
    """ops.set_wgrad_overlap: K5T / K5 run on a side stream that forks from backward and is joined at its end.
    The gradients must be bit-identical to the in-order ones (deterministic kernels), autograd must have installed
    the deferred tensors as .grad by reference (a clone would read them before their kernel ran), a weight that
    already holds a .grad must not be deferred, and the whole step must survive a CUDA-graph capture."""
    from workloads import resnet_cifar
    torch.manual_seed(3)
    dev = torch.device("cuda:0")
    model = resnet_cifar(20, 10, P.PowerOfTwoQuantizer, 4).to(dev).train()
    P.enable_weight_prefetch(model)
    x = torch.randn(64, 3, 32, 32, device=dev)
    y = torch.randint(0, 10, (64,), device=dev)
    crit = nn.CrossEntropyLoss()
    qconvs = [m for m in model.modules() if isinstance(m, P.QuantizedConv2d)]

    def grads(overlap, accumulate=False):
        ops.set_wgrad_overlap(overlap)
        ops._wgrad_trace = []
        try:
            model.zero_grad(set_to_none=True)
            crit(model(x), y).backward()
            first = list(ops._wgrad_trace)
            if accumulate:
                ops._wgrad_trace = []
                crit(model(x), y).backward()          # .grad exists now: nothing may be deferred
                assert ops._wgrad_trace == []
            torch.cuda.synchronize()
            return [p.grad.clone() for p in model.parameters()], first
        finally:
            ops._wgrad_trace = None
            ops.set_wgrad_overlap(False)

    want, none_deferred = grads(False)
    assert none_deferred == []
    again, _ = grads(False)
    # the plain stem conv's weight gradient is cuDNN's (atomics): compare what is reproducible in order
    stable = [torch.equal(a, b) for a, b in zip(want, again)]
    assert sum(stable) >= len(stable) - 1
    got, deferred = grads(True)
    assert len(deferred) >= len(qconvs) - 2, (len(deferred), len(qconvs))
    ptrs = {m.weight.grad.data_ptr() for m in qconvs}
    assert set(deferred) <= ptrs                      # installed by reference, not cloned
    for ok, a, b in zip(stable, want, got):
        assert torch.equal(a, b) if ok else torch.allclose(a, b, rtol=1e-4, atol=1e-6)
    twice, _ = grads(True, accumulate=True)
    once2, _ = grads(False, accumulate=True)
    for ok, a, b in zip(stable, once2, twice):
        assert torch.equal(a, b) if ok else torch.allclose(a, b, rtol=1e-4, atol=1e-6)

    # the same step inside a CUDA graph: the side stream becomes a parallel branch and is joined before the end
    opt = torch.optim.SGD(model.parameters(), lr=0.0)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    ops.set_wgrad_overlap(True)
    try:
        with torch.cuda.stream(s):
            def step():
                opt.zero_grad(set_to_none=True)
                crit(model(x), y).backward()
                opt.step()
            for _ in range(3):
                step()
            s.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                step()
            for _ in range(3):
                g.replay()
            s.synchronize()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        for ok, a, p in zip(stable, want, model.parameters()):
            assert torch.equal(a, p.grad) if ok else torch.allclose(a, p.grad, rtol=1e-4, atol=1e-6)
    finally:
        ops.set_wgrad_overlap(False)


@pytest.mark.parametrize("momentum,wd", [(0.9, 1e-4), (0.0, 1e-4), (0.9, 0.0), (0.0, 0.0)])
def test_multi_tensor_sgd_is_torch_sgd_bit_for_bit(momentum, wd):
    """optim.SGD.step() = po2_sgd_step (one launch per 96 tensors) against torch.optim.SGD (train.py:54-56) over four
    steps: parameters and momentum buffers bit-identical, state_dict interchangeable; ragged sizes, > 96 tensors,
    a tensor larger than one CTA's chunk, an unaligned view-free odd size, and a parameter without a gradient."""
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(11)
    sizes = [1, 3, 16, 17, 64, 2304, 4095, 4096, 4097, 36864, 70001] + [5 + 7 * i for i in range(100)]
    base = [torch.randn(n, generator=g) for n in sizes]
    a = [torch.nn.Parameter(t.clone().to(dev)) for t in base] + [torch.nn.Parameter(torch.ones(4, device=dev))]
    b = [torch.nn.Parameter(t.clone().to(dev)) for t in base] + [torch.nn.Parameter(torch.ones(4, device=dev))]
    oa = P.optim.SGD(a, lr=0.1, momentum=momentum, weight_decay=wd)
    ob = torch.optim.SGD(b, lr=0.1, momentum=momentum, weight_decay=wd)
    before = ops.LAUNCHES
    for step in range(4):
        for pa, pb in zip(a[:-1], b[:-1]):
            gr = torch.randn(pa.shape, generator=g).to(dev) * (10.0 ** (step - 2))
            pa.grad = gr.clone()
            pb.grad = gr.clone()
        oa.step()
        ob.step()
        if step == 1:                                    # a scheduler changed the rate
            for o in (oa, ob):
                o.param_groups[0]["lr"] = 0.037
    torch.cuda.synchronize()
    assert ops.LAUNCHES - before == 4 * 2                # 111 tensors: two launches per step
    for pa, pb in zip(a, b):
        assert torch.equal(pa, pb)
        if momentum:
            sa, sb = oa.state[pa].get("momentum_buffer"), ob.state[pb].get("momentum_buffer")
            assert (sa is None) == (sb is None)
            if sa is not None:
                assert torch.equal(sa, sb)
    # in-place semantics: the version counters moved like torch's (the weight prefetch keys on them)
    assert all(pa._version == pb._version for pa, pb in zip(a[:-1], b[:-1])) and a[0]._version >= 4
    # the state dicts are interchangeable
    ob.load_state_dict(oa.state_dict())
    oa.load_state_dict(ob.state_dict())
    # what the kernel does not take goes to torch's own step: Nesterov here
    c = [torch.nn.Parameter(base[5].clone().to(dev))]
    d = [torch.nn.Parameter(base[5].clone().to(dev))]
    oc = P.optim.SGD(c, lr=0.1, momentum=0.9, nesterov=True)
    od = torch.optim.SGD(d, lr=0.1, momentum=0.9, nesterov=True)
    for _ in range(2):
        c[0].grad = torch.ones_like(c[0])
        d[0].grad = torch.ones_like(d[0])
        oc.step()
        od.step()
    assert torch.equal(c[0], d[0])


def test_weights_are_requantized_after_the_multi_tensor_sgd_step():
    """The prefetch quantizes a layer again only when its weight's version changed: optim.SGD must bump it (it writes
    through raw pointers).  After a step the prefetched quantized weight has to be Q(new weight), in eager mode and
    inside a captured step."""
    from workloads import resnet_cifar
    torch.manual_seed(4)
    dev = torch.device("cuda:0")
    model = resnet_cifar(20, 10, P.PowerOfTwoQuantizer, 4).to(dev).train()
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

    def check():
        model(x)                                             # the forward pre-hook prefetches
        torch.cuda.synchronize()
        want = P.PowerOfTwoQuantizer.forward(None, conv.weight.detach(), bits=4)
        assert torch.equal(conv.__dict__["_po2_prefetch"].qw, want)

    for _ in range(3):
        step()
        check()
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
        assert not torch.equal(before, conv.weight)          # the captured optimizer step moves the weights ...
        g.replay()
        s.synchronize()
    torch.cuda.current_stream().wait_stream(s)
    # ... and the captured forward quantized the weights it started from: compare with the last replay's input weights
    w_before_last = conv.weight.detach().clone()
    with torch.cuda.stream(s):
        g.replay()
        s.synchronize()
    torch.cuda.synchronize()
    want = P.PowerOfTwoQuantizer.forward(None, w_before_last, bits=4)
    assert torch.equal(conv.__dict__["_po2_prefetch"].qw, want)


def test_eval_after_more_training_sees_the_new_running_statistics_and_weights():
    """Caches keyed on Tensor._version (folded eval-mode norms, prefetched operands) must not survive updates that our
    kernels make through raw pointers: train -> eval (folded) -> train -> eval again has to match the unfolded
    evaluation each time; after graph replays (no Python runs, no version moves) invalidate_caches() does it."""
    from workloads import resnet_cifar
    torch.manual_seed(6)
    dev = torch.device("cuda:0")
    model = resnet_cifar(20, 10, P.PowerOfTwoQuantizer, 4).to(dev)
    P.enable_weight_prefetch(model)
    opt = P.optim.SGD(model.parameters(), lr=0.2, momentum=0.9)
    x = torch.randn(32, 3, 32, 32, device=dev)
    y = torch.randint(0, 10, (32,), device=dev)
    crit = nn.CrossEntropyLoss()

    def step():
        model.train()
        opt.zero_grad(set_to_none=True)
        crit(model(x), y).backward()
        opt.step()

    def evals():
        model.eval()
        with torch.no_grad():
            folded = model(x)
            os.environ["PO2_FOLD_BN"] = "0"
            try:
                plain = model(x)
            finally:
                os.environ.pop("PO2_FOLD_BN", None)
        return folded, plain

    for _ in range(3):
        step()
        step()
        folded, plain = evals()
        assert ((folded - plain).abs().max() / plain.abs().max()).item() < 1e-3
    # a captured step replayed: versions do not move, so the caches must be dropped by hand
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            step()
        s.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            step()
        for _ in range(4):
            g.replay()
        s.synchronize()
    torch.cuda.current_stream().wait_stream(s)
    assert P.invalidate_caches(model) > 0
    folded, plain = evals()
    assert ((folded - plain).abs().max() / plain.abs().max()).item() < 1e-3
    # and the quantized weights the evaluation used are those of the current master weights
    conv = [m for m in model.modules() if isinstance(m, P.QuantizedConv2d)][2]
    assert torch.equal(conv.__dict__["_po2_prefetch"].qw, P.PowerOfTwoQuantizer.forward(None, conv.weight.detach(), bits=4))
