"""FusedSyncBatchNorm (csrc/po2_bn.cu) against torch's own batch norm -- what the reference's
nn.SyncBatchNorm layers (models/resnet.py:38-61) compute -- in fp64 on the CPU.

Tolerance: fp32 elementwise work on fp32 statistics accumulated in double: rel 1e-5 (the
fp32-accumulate bar of BASELINE.json's north_star)."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

TOL = 1e-5


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-30)).item()


def _ref_forward_backward(x, res, w, b, relu, go, eps=1e-5):
    """fp64 CPU reference: returns y, dx, dres, dw, db, batch mean, biased var"""
    xd = x.detach().double().cpu().requires_grad_(True)
    rd = res.detach().double().cpu().requires_grad_(True) if res is not None else None
    wd = w.detach().double().cpu().requires_grad_(True)
    bd = b.detach().double().cpu().requires_grad_(True)
    y = F.batch_norm(xd, None, None, wd, bd, True, 0.0, eps)
    if rd is not None:
        y = y + rd
    if relu:
        y = F.relu(y)
    y.backward(go.detach().double().cpu())
    dims = [0] + list(range(2, xd.dim()))
    return y, xd.grad, rd.grad if rd is not None else None, wd.grad, bd.grad, xd.mean(dims), xd.var(dims, unbiased=False)


SHAPES = [(128, 16, 32, 32), (128, 32, 16, 16), (128, 64, 8, 8), (16, 3, 5, 7), (9, 130, 3, 3), (64, 960, 1, 1),
          (2, 8, 1, 1), (5, 24, 6, 6), (128, 16, 32, 32)]


@pytest.mark.parametrize("shape", SHAPES[:8], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("relu,with_res", [(False, False), (True, False), (True, True), (False, True)])
def test_train_forward_backward_matches_torch_fp64(shape, relu, with_res):
    import po2_quantization_b200 as P
    g = torch.Generator(device="cuda").manual_seed(sum(shape))
    x = (torch.randn(shape, device="cuda", generator=g) * 1.7 + 0.6).requires_grad_(True)
    res = torch.randn(shape, device="cuda", generator=g).requires_grad_(True) if with_res else None
    bn = P.FusedSyncBatchNorm(shape[1]).cuda().train()
    with torch.no_grad():
        bn.weight.copy_(torch.randn(shape[1], generator=torch.Generator().manual_seed(1)) * 0.5 + 1.0)
        bn.bias.copy_(torch.randn(shape[1], generator=torch.Generator().manual_seed(2)) * 0.3)
    go = torch.randn(shape, device="cuda", generator=g)
    y = bn(x, res, relu)
    y.backward(go)
    yr, dxr, drr, dwr, dbr, mean, var = _ref_forward_backward(x, res, bn.weight, bn.bias, relu, go)
    assert _rel(y, yr) < TOL
    n = x.numel() // shape[1]
    if n >= 8:          # with 2 values per channel dx is eps-sized cancellation noise on any implementation
        assert _rel(x.grad, dxr) < 5 * TOL
    else:
        assert (x.grad.double().cpu() - dxr).abs().max().item() < 1e-6
    assert _rel(bn.weight.grad, dwr) < 5 * TOL and _rel(bn.bias.grad, dbr) < 5 * TOL
    if with_res:
        assert _rel(res.grad, drr) < TOL
    assert _rel(bn.running_mean, 0.1 * mean) < TOL
    assert _rel(bn.running_var, 0.9 + 0.1 * var * n / (n - 1)) < TOL
    assert bn.num_batches_tracked.item() == 1


def test_statistics_survive_large_mean():
    """|mean| >> std: shifted sums keep the variance accurate (E[x^2]-E[x]^2 in fp32 would not)."""
    import po2_quantization_b200 as P
    g = torch.Generator(device="cuda").manual_seed(3)
    x = torch.randn(64, 8, 16, 16, device="cuda", generator=g) * 0.01 + 300.0
    bn = P.FusedSyncBatchNorm(8).cuda().train()
    y = bn(x)
    ref = F.batch_norm(x.double().cpu(), None, None, bn.weight.double().cpu(), bn.bias.double().cpu(), True, 0.0, bn.eps)
    assert _rel(y, ref) < 2e-3          # x itself carries only ~3e-5/0.01 relative precision around its mean
    var = x.double().var(dim=(0, 2, 3), unbiased=False).mean().item()
    assert abs(y.std().item() - (var / (var + bn.eps)) ** 0.5) < 1e-3


def test_matches_stock_module_state_and_eval_mode():
    import po2_quantization_b200 as P
    torch.manual_seed(4)
    stock = nn.BatchNorm2d(24).cuda().train()
    mine = P.FusedSyncBatchNorm(24).cuda().train()
    assert set(stock.state_dict()) == set(mine.state_dict())
    mine.load_state_dict(stock.state_dict())
    for it in range(3):
        x = torch.randn(32, 24, 8, 8, device="cuda") * (1 + it) + it
        assert _rel(mine(x), stock(x)) < TOL
    for k, v in stock.state_dict().items():
        assert _rel(mine.state_dict()[k].float(), v.float()) < TOL, k
    stock.eval(), mine.eval()
    x = torch.randn(32, 24, 8, 8, device="cuda")
    res = torch.randn_like(x)
    with torch.no_grad():
        assert _rel(mine(x), stock(x)) < TOL
        assert _rel(mine(x, res, True), F.relu(stock(x) + res)) < TOL
    # eval mode under autograd: the stock path, still correct and differentiable
    x.requires_grad_(True)
    out = mine(x, res, True)
    out.sum().backward()
    assert _rel(out, F.relu(stock(x) + res)) < TOL and x.grad is not None


def test_two_rank_statistics_combine_like_sync_batchnorm():
    """The multi-rank algebra on one GPU: statistics of two half-batches combined by bn_apply and the
    summed backward partials must equal batch norm over the whole batch (what SyncBatchNorm does)."""
    from po2_quantization_b200 import batchnorm as bnm
    g = torch.Generator(device="cuda").manual_seed(5)
    shape = (24, 16, 8, 8)
    x = torch.randn(shape, device="cuda", generator=g) * 2 + 1
    x[:10] += 3.0                                             # the two "ranks" see different distributions
    go = torch.randn(shape, device="cuda", generator=g)
    w = torch.rand(16, device="cuda", generator=g) + 0.5
    b = torch.randn(16, device="cuda", generator=g)
    parts = [(x[:10].contiguous(), go[:10].contiguous()), (x[10:].contiguous(), go[10:].contiguous())]
    C = 16
    stats = torch.empty(2, 2 * C + 1, device="cuda")
    for r, (xr, _) in enumerate(parts):
        bnm.bn_stats_out(xr, stats[r])
    ys, dxs, sums, saves = [], [], [], []
    for xr, _ in parts:
        y = torch.empty_like(xr)
        sm, si = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
        bnm.bn_apply_out(xr, None, y, stats, w, b, None, None, None, 0.1, 1e-5, True, False, sm, si)
        ys.append(y), saves.append((sm, si))
    for (xr, gr), y, (sm, si) in zip(parts, ys, saves):
        s = torch.empty(2 * C, device="cuda")
        bnm.bn_bwd_reduce_out(gr, xr, y, sm, si, s, None, None, True)
        sums.append(s)
    total = sums[0] + sums[1]                                  # the all_reduce
    for (xr, gr), y, (sm, si) in zip(parts, ys, saves):
        dx = torch.empty_like(xr)
        bnm.bn_bwd_apply_out(gr, xr, y, sm, si, w, total, stats, dx, None, True)
        dxs.append(dx)
    yr, dxr, _, _, _, _, _ = _ref_forward_backward(x, None, w, b, True, go)
    assert _rel(torch.cat(ys), yr) < TOL
    assert _rel(torch.cat(dxs), dxr) < 5 * TOL


def test_peer_exchange_protocol_two_ranks_emulated_on_one_gpu():
    """The mailbox protocol (publish into every rank's mailbox, epoch flags, slot rotation) with both
    "ranks" on one device: producers of both ranks are enqueued before the consumers, so nothing has to
    spin.  Six exchanges (> BN_SLOTS) so slots get reused.  Real cross-GPU runs: tools/check_sync_bn.py."""
    from po2_quantization_b200 import _lib, batchnorm as bnm
    g = torch.Generator(device="cuda").manual_seed(11)
    C, shape = 24, (20, 24, 6, 6)
    boxes = [torch.zeros(int(_lib.load().po2_bn_mailbox_bytes()), dtype=torch.uint8, device="cuda") for _ in range(2)]
    ptrs = [b.data_ptr() for b in boxes]
    ex = [bnm.PeerExchange(ptrs, r, 2) for r in range(2)]
    w = torch.rand(C, device="cuda", generator=g) + 0.5
    b = torch.randn(C, device="cuda", generator=g)
    for it in range(3):
        x = torch.randn(shape, device="cuda", generator=g) * (1 + it) + it
        go = torch.randn(shape, device="cuda", generator=g)
        parts = [(x[:8].contiguous(), go[:8].contiguous()), (x[8:].contiguous(), go[8:].contiguous())]
        stat = [torch.empty(2 * C + 1, device="cuda") for _ in range(2)]
        for r in range(2):
            bnm.bn_stats_out(parts[r][0], stat[r], ex[r])
        ys, saves, dense = [], [], []
        for r in range(2):
            y = torch.empty_like(parts[r][0])
            sm, si = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
            d = torch.empty(2, 2 * C + 1, device="cuda")
            bnm.bn_apply_out(parts[r][0], None, y, None, w, b, None, None, None, 0.1, 1e-5, True, False, sm, si,
                             exch=ex[r], stats_dense=d)
            ys.append(y), saves.append((sm, si)), dense.append(d)
        assert torch.equal(dense[0], dense[1]) and torch.equal(dense[0][0], stat[0]) and torch.equal(dense[0][1], stat[1])
        sums = [torch.empty(2 * C, device="cuda") for _ in range(2)]
        for r in range(2):
            bnm.bn_bwd_reduce_out(parts[r][1], parts[r][0], ys[r], *saves[r], sums[r], None, None, True, ex[r])
        dxs = []
        for r in range(2):
            dx = torch.empty_like(parts[r][0])
            bnm.bn_bwd_apply_out(parts[r][1], parts[r][0], ys[r], *saves[r], w, None, dense[r], dx, None, True, ex[r])
            dxs.append(dx)
        yr, dxr, *_ = _ref_forward_backward(x, None, w, b, True, go)
        assert _rel(torch.cat(ys), yr) < TOL, it
        assert _rel(torch.cat(dxs), dxr) < 5 * TOL, it
    for bx in boxes:
        assert bx[0:4].view(torch.int32).item() == 6 and bx[4:8].view(torch.int32).item() == 0   # epoch, error flag


def test_cuda_graph_capture_and_replay():
    import po2_quantization_b200 as P
    bn = P.FusedSyncBatchNorm(32).cuda().train()
    x = torch.randn(16, 32, 8, 8, device="cuda", requires_grad=True)
    res = torch.randn(16, 32, 8, 8, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            bn(x, res, True).sum().backward()
        x.grad = None
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, stream=s):
            y = bn(x, res, True)
            y.sum().backward()
    torch.cuda.current_stream().wait_stream(s)
    nb = bn.num_batches_tracked.item()
    with torch.no_grad():
        x.copy_(torch.randn_like(x) * 3)
    gr.replay()
    torch.cuda.synchronize()
    yr, dxr, *_ = _ref_forward_backward(x, res, bn.weight, bn.bias, True, torch.ones_like(x))
    assert _rel(y, yr) < TOL and _rel(x.grad, dxr) < 5 * TOL
    assert bn.num_batches_tracked.item() == nb + 1


def test_resnet20_train_step_with_fused_norm_equals_stock_norm():
    """Same model, same weights: FusedSyncBatchNorm vs nn.SyncBatchNorm in the block graph."""
    import po2_quantization_b200 as P
    from po2_quantization_b200 import ops
    from workloads import resnet_cifar
    torch.manual_seed(6)
    ops.set_conv_mode("fp32")
    ops.set_dgrad_mode("aten")
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        a = resnet_cifar(20, 10, P.PowerOfTwoQuantizer, 4).cuda().train()
        b = resnet_cifar(20, 10, P.PowerOfTwoQuantizer, 4, norm_cls=nn.SyncBatchNorm).cuda().train()
        b.load_state_dict(a.state_dict())
        x = torch.randn(32, 3, 32, 32, device="cuda")
        t = torch.randint(0, 10, (32,), device="cuda")
        la = F.cross_entropy(a(x), t)
        lb = F.cross_entropy(b(x), t)
        la.backward(), lb.backward()
        assert abs(la.item() - lb.item()) < 1e-4
        pb = dict(b.named_parameters())
        for n, p in a.named_parameters():
            gb = pb[n].grad
            if gb.abs().max() < 1e-6:
                continue
            assert _rel(p.grad, gb) < 2e-2, n                  # train-mode BN chains amplify fp32 rounding
        for (n, va), vb in zip(a.state_dict().items(), b.state_dict().values()):
            if "running" in n:
                assert _rel(va, vb) < 1e-4, n
    finally:
        ops.set_conv_mode(ops.DEFAULT_CONV_MODE)
        ops.set_dgrad_mode("tc")
        torch.backends.cudnn.allow_tf32 = old


@pytest.mark.parametrize("act", ["relu6", "silu"])
@pytest.mark.parametrize("shape", [(32, 24, 8, 8), (16, 96, 3, 3), (64, 160, 1, 1)], ids=lambda s: "x".join(map(str, s)))
def test_activation_variants_match_torch(act, shape):
    """ReLU6 (MobileNetV2) and SiLU (MobileViT) behind the norm: train mode with backward (SiLU through
    F.silu behind the kernel), and the fully fused eval / no-grad path."""
    import po2_quantization_b200 as P
    g = torch.Generator(device="cuda").manual_seed(sum(shape))
    fn = {"relu6": F.relu6, "silu": F.silu}[act]
    x = (torch.randn(shape, device="cuda", generator=g) * 2.5 + 0.5).requires_grad_(True)
    go = torch.randn(shape, device="cuda", generator=g)
    bn = P.FusedSyncBatchNorm(shape[1], act=act).cuda().train()
    with torch.no_grad():
        bn.weight.copy_(torch.rand(shape[1], device="cuda", generator=g) * 2 + 1)     # large gamma: ReLU6 clips at both ends
        bn.bias.copy_(torch.randn(shape[1], device="cuda", generator=g) + 1)
    y = bn(x)
    y.backward(go)
    xd = x.detach().double().cpu().requires_grad_(True)
    yr = fn(F.batch_norm(xd, None, None, bn.weight.detach().double().cpu(), bn.bias.detach().double().cpu(), True, 0.0, bn.eps))
    yr.backward(go.double().cpu())
    assert _rel(y, yr) < TOL
    n = x.numel() // shape[1]
    if n >= 64:
        assert _rel(x.grad, xd.grad) < 1e-4
    bn.eval()
    with torch.no_grad():
        ye = bn(x.detach())
        ref = fn(F.batch_norm(x.detach().double().cpu(), bn.running_mean.double().cpu(), bn.running_var.double().cpu(),
                              bn.weight.double().cpu(), bn.bias.double().cpu(), False, 0.0, bn.eps))
    assert _rel(ye, ref) < TOL


@pytest.mark.parametrize("fused", ["1", "0"], ids=["one_launch", "reduce_apply"])
@pytest.mark.parametrize("shape", [(16, 32, 16, 16), (8, 24, 6, 6), (16, 96, 3, 3)], ids=lambda s: "x".join(map(str, s)))
def test_silu_backward_runs_in_the_norm_kernels(shape, fused, monkeypatch):
    """conv-norm-SiLU (models/mobile_vit.py:16-22) under autograd: the SiLU slope is applied inside the backward
    kernels (one-launch and reduce + apply forms, 128-bit and scalar paths), no separate F.silu pass; dx, dgamma and
    dbeta against fp64 autograd.  Behind a residual add the activation stays a separate F.silu."""
    import po2_quantization_b200 as P
    from po2_quantization_b200 import ops
    monkeypatch.setenv("PO2_BN_FUSED", fused)
    g = torch.Generator(device="cuda").manual_seed(sum(shape) + 5)
    x = (torch.randn(shape, device="cuda", generator=g) * 1.5 - 0.3).requires_grad_(True)
    go = torch.randn(shape, device="cuda", generator=g)
    bn = P.FusedSyncBatchNorm(shape[1], act="silu").cuda().train()
    with torch.no_grad():
        bn.weight.copy_(torch.rand(shape[1], device="cuda", generator=g) + 0.5)
        bn.bias.copy_(torch.randn(shape[1], device="cuda", generator=g) * 0.5)
    before = ops.LAUNCHES
    y = bn(x)
    y.backward(go)
    torch.cuda.synchronize()
    one_launch = fused == "1" and (shape[2] * shape[3]) % 4 == 0          # the one-launch forms are 128-bit only
    assert ops.LAUNCHES - before == (2 if one_launch else 4)
    xd = x.detach().double().cpu().requires_grad_(True)
    wd = bn.weight.detach().double().cpu().requires_grad_(True)
    bd = bn.bias.detach().double().cpu().requires_grad_(True)
    yr = F.silu(F.batch_norm(xd, None, None, wd, bd, True, 0.0, bn.eps))
    yr.backward(go.double().cpu())
    assert _rel(y, yr) < TOL
    assert _rel(x.grad, xd.grad) < 1e-4
    assert _rel(bn.weight.grad, wd.grad) < 1e-4
    assert _rel(bn.bias.grad, bd.grad) < 1e-4
    # SiLU behind a residual add: norm + add in the kernel, F.silu behind it, same numbers
    x2 = x.detach().clone().requires_grad_(True)
    r2 = torch.randn(shape, device="cuda", generator=g).requires_grad_(True)
    bn.zero_grad()
    bn(x2, residual=r2).backward(go)
    xd2 = x.detach().double().cpu().requires_grad_(True)
    rd2 = r2.detach().double().cpu().requires_grad_(True)
    F.silu(F.batch_norm(xd2, None, None, wd.detach(), bd.detach(), True, 0.0, bn.eps) + rd2).backward(go.double().cpu())
    assert _rel(x2.grad, xd2.grad) < 1e-4
    assert _rel(r2.grad, rd2.grad) < 1e-4


def test_mobilenet_and_mobilevit_fused_norm_state_dict_and_forward():
    """The fused-norm variants of the MobileNetV2 / MobileViT workloads keep the stock state_dict keys
    and compute the same eval-mode forward."""
    from po2_quantization_b200 import ops
    from workloads import mobilenet_v2_cifar, mobilevit_xs
    torch.manual_seed(3)
    ops.set_conv_mode("fp32")            # keep bf16 / TF32 activation rounding out of a norm-vs-norm comparison
    old_tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        for build in (lambda f: mobilenet_v2_cifar(10, None, 4, fused_norm=f),
                      lambda f: mobilevit_xs((32, 32), 10, (1, 1), None, 8, fused_norm=f)):
            a, b = build(True).cuda(), build(False).cuda()
            assert list(a.state_dict().keys()) == list(b.state_dict().keys())
            b.load_state_dict(a.state_dict())
            x = torch.randn(16, 3, 32, 32, device="cuda")
            a.train(), b.train()             # one train-mode pass for non-trivial running statistics
            with torch.no_grad():
                a(x), b(x)
            a.eval(), b.eval()
            with torch.no_grad():
                ya, yb = a(x), b(x)
            assert _rel(ya, yb.double()) < 1e-3, _rel(ya, yb.double())
    finally:
        ops.set_conv_mode(ops.DEFAULT_CONV_MODE)
        torch.backends.cudnn.allow_tf32 = old_tf32


def test_skip_connection_gradient_is_added_inside_the_norm_kernels(monkeypatch):
    """A residual block's input receives two gradients: the conv branch's and the skip connection's.  With the
    FusedSyncBatchNorm modules of workloads/resnet_cifar.py the second one is left at the producing norm's autograd
    node (_SkipGrad) and added inside that norm's backward kernels (dy + dy2) instead of by an accumulation kernel:
    same fp32 addition, so every gradient is bit-identical, with one launch less per identity block.  Both backward
    forms (one launch, reduce + apply)."""
    import po2_quantization_b200 as P
    from po2_quantization_b200 import ops
    from workloads import resnet_cifar
    torch.manual_seed(5)
    model = resnet_cifar(20, 10, P.PowerOfTwoQuantizer, 4).cuda().train()
    P.enable_weight_prefetch(model)
    x = torch.randn(32, 3, 32, 32, device="cuda")
    y = torch.randint(0, 10, (32,), device="cuda")
    crit = torch.nn.CrossEntropyLoss()

    def grads(skip, fused):
        monkeypatch.setenv("PO2_SKIP_GRAD", skip)
        monkeypatch.setenv("PO2_BN_FUSED_BWD", fused)
        model.zero_grad(set_to_none=True)
        crit(model(x), y).backward()
        torch.cuda.synchronize()
        return [p.grad.clone() for p in model.parameters()]

    grads("0", "1")                                          # warm-up: the first forward records the prefetch shapes
    for fused in ("1", "0"):
        want, again, got = grads("0", fused), grads("0", fused), grads("1", fused)
        stable = [torch.equal(a, b) for a, b in zip(want, again)]       # all but the stem conv's cuDNN weight gradient
        assert sum(stable) >= len(stable) - 1
        for ok, a, b in zip(stable, want, got):
            assert torch.equal(a, b) if ok else torch.allclose(a, b, rtol=1e-4, atol=1e-6)
    # a graph that is walked twice (retain_graph): the skip gradient is routed again, gradients accumulate to 2x
    monkeypatch.setenv("PO2_SKIP_GRAD", "1")
    model.zero_grad(set_to_none=True)
    loss = crit(model(x), y)
    loss.backward(retain_graph=True)
    once = [p.grad.clone() for p in model.parameters()]
    loss.backward()
    torch.cuda.synchronize()
    for a, p in zip(once, model.parameters()):
        assert torch.allclose(p.grad, 2 * a, rtol=1e-4, atol=1e-6)
    # the accumulation kernels are gone: count torch's add kernels with the profiler
    from torch.profiler import ProfilerActivity, profile

    def adds(skip):
        monkeypatch.setenv("PO2_SKIP_GRAD", skip)
        monkeypatch.setenv("PO2_BN_FUSED_BWD", "1")
        model.zero_grad(set_to_none=True)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            crit(model(x), y).backward()
            torch.cuda.synchronize()
        return sum(e.count for e in prof.key_averages() if "CUDAFunctor_add" in e.key)
    assert adds("0") - adds("1") == 7                        # ResNet-20: 9 blocks, 7 of them with an identity shortcut
