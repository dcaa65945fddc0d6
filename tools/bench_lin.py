"""lin / lin+ layers on the conv kernels against the stock path (set_conv_mode("cudnn")), on one GPU:

  * ResNet-56 4-bit QAT step (forward + backward + SGD, batch 128, CUDA graph) with lin, lin+ and PO2 weights: the
    kernel path and the stock path timed alternately in one process, three repetitions, median and spread;
  * the lin quantizer alone for the 56 weights of that model: 56 po2_lin_quantize launches against one multi-tensor
    po2_lin_quantize_pack_multi launch (CUDA events; the 3.4 MB of weights stay resident in L2 between passes);
  * ResNet-20 and MobileNetV2 lin+ 4-bit PTQ eval forward (batch 256, CUDA graph), with and without fold_conv_bn.

The card's name and power limit are read in the same process and written beside the numbers.

    python tools/bench_lin.py [--out profiles/r03_lin_bench.json]
"""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn as nn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import po2_quantization_b200 as P  # noqa: E402
from po2_quantization_b200 import _lib, ops  # noqa: E402
from workloads import mobilenet_v2_cifar, resnet_cifar  # noqa: E402

QUANT = {"lin": P.LinearPowerOfTwoQuantizer, "lin+": P.LinearPowerOfTwoPlusQuantizer, "po2": P.PowerOfTwoQuantizer}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def capture(fn, warmup=3):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(warmup):
            fn()
        s.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    return g


def replay_ms(g, iters):
    for _ in range(3):
        g.replay()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def qat_step(quantize_fn, mode):
    """(graph, step, model): the ResNet-56 step as bench.build_training builds it, captured under conv mode `mode`.
    The graph replays into the memory of the model, the optimizer state and the batch: keep `step`, which holds
    them, alive as long as the graph."""
    ops.set_conv_mode(mode)
    torch.manual_seed(8)
    dev = torch.device("cuda:0")
    model = resnet_cifar(56, 10, quantize_fn, 4).to(dev).train()
    P.enable_weight_prefetch(model)
    ops.set_wgrad_overlap(True)
    opt = P.optim.SGD(model.parameters(), lr=0.1, momentum=0.9, weight_decay=1e-4)
    crit = nn.CrossEntropyLoss()
    x = torch.randn(128, 3, 32, 32, device=dev)
    t = torch.randint(0, 10, (128,), device=dev)

    def step():
        opt.zero_grad(set_to_none=True)
        crit(model(x), t).backward()
        opt.step()

    g = capture(step)
    ops.set_conv_mode(ops.DEFAULT_CONV_MODE)
    return g, step, model


def bench_qat(iters=100, reps=3):
    out = {}
    for name, q in QUANT.items():
        arms = {"kernels_tf32": qat_step(q, "tf32"), "stock_cudnn": qat_step(q, "cudnn")}
        ms = {k: [] for k in arms}
        for _ in range(reps):
            for k, arm in arms.items():               # alternately, in one process
                ms[k].append(replay_ms(arm[0], iters))
        out[name] = {k: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v), "runs_ms": v}
                     for k, v in ms.items()}
        out[name]["speedup_stock_over_kernels"] = out[name]["stock_cudnn"]["median_ms"] / out[name]["kernels_tf32"]["median_ms"]
        del arms
        torch.cuda.synchronize()
    return out


def bench_quantizer(iters=200):
    """56 single-tensor launches against one multi-tensor launch, same weights (lin+ 4-bit, ResNet-56)"""
    _g, _step, model = qat_step(P.LinearPowerOfTwoPlusQuantizer, "tf32")
    lib = _lib.load()
    convs = [m for m in model.modules() if isinstance(m, P.QuantizedConv2d)]
    ys = [torch.empty_like(m.weight) for m in convs]
    st = ops._stream_ptr(torch.device("cuda:0"))

    def singles():
        for m, y in zip(convs, ys):
            K, C, R, S = m.weight.shape
            _lib.check(lib.po2_lin_quantize(m.weight.data_ptr(), y.data_ptr(), K, C, R * S, 4, ops.LIN_ITERS, 1, ops._flavor,
                                            st), "po2_lin_quantize")

    from po2_quantization_b200 import prefetch
    tab = [t for k, t in prefetch._tables.items() if isinstance(k, tuple) and k[1] == "lin"][-1]

    def multi():
        _lib.check(lib.po2_lin_quantize_pack_multi(tab.dev.data_ptr(), tab.n, tab.csize[0], tab.csize[1], st),
                   "po2_lin_quantize_pack_multi")

    res = {"layers": len(convs), "multi_tensors": tab.n, "multi_ctas": tab.csize[0],
           "weight_bytes": sum(m.weight.numel() * 4 for m in convs),
           "l2_state": "warm: the weights, y and the packed operands (a few MB) stay in the 126 MB L2 between passes"}
    for name, fn in (("single_x56_us", singles), ("multi_x1_us", multi)):
        for _ in range(5):
            fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        res[name] = a.elapsed_time(b) * 1000.0 / iters
    return res


def bench_ptq(batch=256, iters=50):
    out = {}
    x = torch.randn(batch, 3, 32, 32, device="cuda")
    for name, build in (("resnet20", lambda: resnet_cifar(20, 10, None, 4)), ("mobilenetv2", lambda: mobilenet_v2_cifar(10, None, 4))):
        torch.manual_seed(3)
        base = build().cuda()
        P.quantize_model(base, P.LinearPowerOfTwoPlusQuantizer, 4)
        base.eval()
        row = {}
        for fold in (False, True):
            for mode in ("tf32", "cudnn"):
                m = copy.deepcopy(base)
                if fold:
                    P.fold_conv_bn(m)
                ops.set_conv_mode(mode)
                with torch.no_grad():
                    g = capture(lambda: m(x))
                    row[f"{'fold' if fold else 'nofold'}_{mode}_ms"] = replay_ms(g, iters)
                ops.set_conv_mode(ops.DEFAULT_CONV_MODE)
        out[name] = row
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r03_lin_bench.json")
    ap.add_argument("--iters", type=int, default=100)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_lin.py measures on a CUDA device; none is visible")
    res = {"card": card(), "qat_step_resnet56_b128_4bit": bench_qat(a.iters), "quantizer_resnet56_lin_plus_4bit": bench_quantizer(),
           "ptq_eval_forward_lin_plus_4bit_b256": bench_ptq()}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
