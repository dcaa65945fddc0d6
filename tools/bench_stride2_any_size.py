"""Backward of the odd-size stride-2 layers on our kernels (po2_dilate2_into + the stride-1 gradient kernels) against
the route they took before, aten.convolution_backward, on one GPU:

  * per layer: the 3x3 depthwise stride-2 layers onto a 1x1 map of MobileNetV2-CIFAR (576 channels, 2x2 -> 1x1,
    batch 128) and MobileViT-xs at 32x32 (320 channels, batch 16): the data and the weight gradient, i.e.
    ops._conv_backward (zero-insertion + depthwise data gradient + depthwise weight gradient) against
    aten.convolution_backward computing both.  Each arm is 200 calls captured in one CUDA graph and timed with CUDA
    events over the replay, after warm-up; the operands are the same in every call (L2-resident);
  * the PO2+ 4-bit QAT step (forward + backward + optim.SGD, CUDA graph, weight prefetch, weight gradients on the
    side stream) of MobileNetV2-CIFAR (batch 128) and MobileViT-xs at 32x32 (batch 16): every layer on our kernels,
    against the same step with the backward of the stride-2 layers that po2_dilate2 refuses sent to
    aten.convolution_backward (what ops._conv_backward did for them before).  Two graphs per arm, timed
    alternately in one process, five repetitions each, median and spread over both graphs of an arm.

The card's name and power limit are read in the same process and written beside the numbers.

    python tools/bench_stride2_any_size.py [--out profiles/r06_stride2_any_size.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn as nn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import po2_quantization_b200 as P  # noqa: E402
from po2_quantization_b200 import ops  # noqa: E402
from workloads import mobilenet_v2_cifar, mobilevit_xs  # noqa: E402

# (model, channels, H == W, batch)
LAYERS = [("mobilenetv2", 576, 2, 128), ("mobilevit_xs32", 320, 2, 16)]


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


def _odd_stride2(stride, x, g):
    return stride == 2 and bool(x.shape[2] % 2 or x.shape[3] % 2 or g.shape[3] % 2)


def _aten_backward(g, x, w, stride, pad, groups, need_x, need_w):
    gx, gw, _ = torch.ops.aten.convolution_backward(g.contiguous(), x.contiguous(), w, None, [stride, stride], [pad, pad],
                                                    [1, 1], False, [0, 0], groups, [need_x, need_w, False])
    return gx, gw


def bench_layers(calls=200, reps=5):
    torch.backends.cudnn.allow_tf32 = True
    out = []
    for model, C, HW, B in LAYERS:
        x = torch.randn(B, C, HW, HW, device="cuda")
        w0 = torch.randn(C, 1, 3, 3, device="cuda") * 0.1
        w, codes, scale, zc, sse = torch.ops.po2.quantize_full(w0, 4, 1, True)
        PQ = (HW - 1) // 2 + 1
        g = torch.randn(B, C, PQ, PQ, device="cuda")
        row = {"model": model, "layer": f"depthwise 3x3 stride 2, {C} channels, {HW}x{HW} -> {PQ}x{PQ}", "batch": B}

        def ours():
            for _ in range(calls):
                ops._conv_backward(g, x, w, scale, 2, 1, C, 2, True, True)

        def aten():
            for _ in range(calls):
                _aten_backward(g, x, w, 2, 1, C, True, True)

        gx, gw = ops._conv_backward(g, x, w, scale, 2, 1, C, 2, True, True)
        rx, rw = _aten_backward(g.double(), x.double(), w.double(), 2, 1, C, True, True)
        row["rel_err_vs_fp64"] = {"dx": ((gx.double() - rx).abs().max() / rx.abs().max()).item(),
                                  "dw": ((gw.double() - rw).abs().max() / rw.abs().max()).item()}
        graphs = {"po2_kernels_us": capture(ours, warmup=1), "aten_cudnn_us": capture(aten, warmup=1)}
        ts = {k: [] for k in graphs}
        for _ in range(reps):
            for k, gr in graphs.items():                 # alternately
                ts[k].append(replay_ms(gr, 5) * 1000.0 / calls)
        for k, v in ts.items():
            row[k] = statistics.median(v)
            row[k.replace("_us", "_spread_us")] = [min(v), max(v)]
        row["speedup_over_aten"] = row["aten_cudnn_us"] / row["po2_kernels_us"]
        out.append(row)
        print(json.dumps(row), flush=True)
        del graphs
    return out


def qat_step(name, aten_route):
    """(graph, step): the PO2+ 4-bit QAT step of `name`, captured with the odd-size stride-2 backward on our kernels or
    on aten.convolution_backward.  Keep `step`, which holds the model, the optimizer state and the batch, alive as long
    as the graph."""
    torch.manual_seed(8)
    dev = torch.device("cuda:0")
    if name == "mobilenetv2_b128":
        model, batch = mobilenet_v2_cifar(10, P.PowerOfTwoPlusQuantizer, 4), 128
    else:
        model, batch = mobilevit_xs((32, 32), 10, (1, 1), P.PowerOfTwoPlusQuantizer, 4), 16
    model = model.to(dev).train()
    P.enable_weight_prefetch(model)
    opt = P.optim.SGD(model.parameters(), lr=0.1, momentum=0.9, weight_decay=1e-4)
    crit = nn.CrossEntropyLoss()
    x = torch.randn(batch, 3, 32, 32, device=dev)
    t = torch.randint(0, 10, (batch,), device=dev)

    def step():
        opt.zero_grad(set_to_none=True)
        crit(model(x), t).backward()
        opt.step()

    real, taken = ops._conv_backward, []

    def routed(g, xx, w, scale, stride, pad, groups, compute, need_x, need_w, *args, **kw):
        if aten_route and _odd_stride2(stride, xx, g):
            taken.append(f"{list(xx.shape)} groups {groups}")
            return _aten_backward(g, xx, w, stride, pad, groups, need_x, need_w)
        return real(g, xx, w, scale, stride, pad, groups, compute, need_x, need_w, *args, **kw)

    ops._conv_backward = routed
    try:
        gr = capture(step)
    finally:
        ops._conv_backward = real
    return gr, step, sorted(set(taken))


def bench_steps(iters=100, reps=5):
    """Two graphs per arm, built in the order ours, aten, aten, ours: two captures of the same step can differ by more
    than the route of one small layer does, so each arm's runs are pooled over both of its graphs"""
    torch.backends.cudnn.allow_tf32 = True
    ops.set_wgrad_overlap(True)
    res = {}
    order = (("po2_kernels", False), ("odd_stride2_on_aten", True), ("odd_stride2_on_aten", True), ("po2_kernels", False))
    for name in ("mobilenetv2_b128", "mobilevit_xs32_b16"):
        notes, note = [], ops.note_library_path
        ops.note_library_path = lambda key, message: notes.append(message) if key == "conv_backward_aten" else None
        try:
            graphs = [(arm, qat_step(name, aten)) for arm, aten in order]
        finally:
            ops.note_library_path = note
        per_graph = [[] for _ in graphs]
        for _ in range(reps):
            for i, (arm, built) in enumerate(graphs):      # alternately, in one process
                per_graph[i].append(replay_ms(built[0], iters))
        out = {}
        for arm, _ in order[:2]:
            runs = [t for (a, _), v in zip(graphs, per_graph) if a == arm for t in v]
            out[arm] = {"median_ms": statistics.median(runs), "min_ms": min(runs), "max_ms": max(runs),
                        "per_graph_median_ms": [statistics.median(v) for (a, _), v in zip(graphs, per_graph) if a == arm],
                        "runs_ms": runs}
        out["aten_over_kernels"] = out["odd_stride2_on_aten"]["median_ms"] / out["po2_kernels"]["median_ms"]
        out["layers_on_aten_in_the_aten_arm"] = graphs[1][1][2]
        out["conv_backward_aten_notes"] = sorted(set(notes))        # the library's own fallbacks, both arms
        res[name] = out
        print(name, json.dumps(out), flush=True)
        del graphs
    ops.set_wgrad_overlap(False)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r06_stride2_any_size.json")
    ap.add_argument("--iters", type=int, default=100)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_stride2_any_size.py measures on a CUDA device; none is visible")
    res = {"card": card(), "layers_l2_state": "operands L2-resident: the same x, g and w in every call",
           "layers": bench_layers(), "qat_steps_po2plus_4bit": bench_steps(a.iters)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
