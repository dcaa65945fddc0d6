"""Weight gradient of the wide pointwise layers (conv_wgrad_pw_kernel + conv_wgrad_reduce_kernel, kernel kind 3)
against cuDNN, on one GPU:

  * per layer: the 16 1x1 layer shapes of MobileNetV2-CIFAR (batch 128) and MobileViT-xs 32x32 (batch 16) that the
    tcgen05 weight-gradient kernels do not take (24->144 @8x8 is at the bound B*H*W = 8192), plus one shape at the
    bound B*H*W*C*K = 2^26 and, for reference, shapes beyond the bounds (cuDNN only).  Each arm is 200 calls
    captured in one CUDA graph and timed with CUDA events over the replay; the library call against
    aten.convolution_backward computing the weight gradient only, with TF32 allowed (PyTorch's cuDNN default).
    The same operands are read by every call, so they are L2-resident (a few MB against 126 MB of L2);
  * the MobileNetV2 PO2+ 4-bit QAT step (forward + backward + optim.SGD, batch 128, CUDA graph, weight prefetch,
    weight gradients on the side stream): the default tf32 kernels against set_conv_mode("cudnn"), timed alternately
    in one process, three repetitions, median and spread.

The script uses only the public interface, so the same file runs on an older tree (layers it does not take are
reported as such).  The card's name and power limit are read in the same process and written beside the numbers.

    python tools/bench_pw_wgrad.py [--out profiles/r04_pw_wgrad_bench.json]
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
from po2_quantization_b200 import _lib, ops  # noqa: E402
from workloads import mobilenet_v2_cifar  # noqa: E402

# (model, C, K, H == W, batch)
LAYERS = [("mobilenetv2", C, K, HW, 128) for C, K, HW in
          [(24, 144, 8), (32, 192, 4), (64, 384, 2), (384, 64, 2), (384, 96, 2), (96, 576, 2), (576, 96, 2),
           (576, 160, 1), (160, 960, 1), (960, 160, 1), (960, 320, 1)]] + \
         [("mobilevit_xs32", C, K, HW, 16) for C, K, HW in
          [(48, 192, 8), (64, 256, 4), (80, 320, 2), (320, 96, 1), (96, 144, 1)]] + \
         [("bound_FMA_2^26", 64, 512, 4, 128)] + \
         [("beyond_bound", C, K, HW, B) for C, K, HW, B in [(24, 144, 8, 256), (160, 960, 8, 128)]]


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


def bench_layers(calls=200, reps=3):
    lib = _lib.load()
    torch.backends.cudnn.allow_tf32 = True
    out = []
    for model, C, K, HW, B in LAYERS:
        x = torch.randn(B, C, HW, HW, device="cuda")
        g = torch.randn(B, K, HW, HW, device="cuda")
        w = torch.randn(K, C, 1, 1, device="cuda")
        gw = torch.empty_like(w)
        q = (B, C, HW, HW, K, 1, 1, 1, 0, 1, 2)
        kind = lib.po2_conv2d_wgrad_kernel_kind(*q)
        row = {"model": model, "layer": f"{C}->{K} 1x1 @{HW}x{HW}", "batch": B, "B*H*W": B * HW * HW,
               "fma": B * HW * HW * C * K, "wgrad_kernel_kind": kind}

        def aten():
            for _ in range(calls):
                torch.ops.aten.convolution_backward(g, x, w, None, [1, 1], [0, 0], [1, 1], False, [0, 0], 1,
                                                    [False, True, False])

        arms = {"cudnn_tf32_us": aten}
        if kind != 0:
            ws = torch.empty(int(lib.po2_conv2d_wgrad_workspace(*q)), dtype=torch.uint8, device="cuda")
            row["workspace_bytes"] = ws.numel()

            def ours():
                st = ops._stream_ptr(x.device)
                for _ in range(calls):
                    _lib.check(lib.po2_conv2d_wgrad(g.data_ptr(), x.data_ptr(), gw.data_ptr(), *q, ws.data_ptr(),
                                                    ws.numel(), st), "po2_conv2d_wgrad")

            arms["po2_kernel_us"] = ours
            ref = torch.ops.aten.convolution_backward(g.double(), x.double(), w.double(), None, [1, 1], [0, 0], [1, 1],
                                                      False, [0, 0], 1, [False, True, False])[1]
            ours()
            torch.cuda.synchronize()
            row["rel_err_vs_fp64"] = ((gw.double() - ref).abs().max() / ref.abs().max()).item()
        graphs = {k: capture(fn, warmup=1) for k, fn in arms.items()}
        ts = {k: [] for k in graphs}
        for _ in range(reps):
            for k, gr in graphs.items():                 # alternately
                ts[k].append(replay_ms(gr, 5) * 1000.0 / calls)
        for k, v in ts.items():
            row[k] = statistics.median(v)
            row[k.replace("_us", "_spread_us")] = [min(v), max(v)]
        if "po2_kernel_us" in row:
            row["speedup_over_cudnn"] = row["cudnn_tf32_us"] / row["po2_kernel_us"]
        out.append(row)
        print(json.dumps(row), flush=True)
        del graphs
    return out


def qat_step(mode):
    """(graph, step, model): the MobileNetV2 PO2+ 4-bit QAT step, captured under conv mode `mode`.  Keep `step`, which
    holds the model, the optimizer state and the batch, alive as long as the graph."""
    ops.set_conv_mode(mode)
    torch.manual_seed(8)
    dev = torch.device("cuda:0")
    model = mobilenet_v2_cifar(10, P.PowerOfTwoPlusQuantizer, 4).to(dev).train()
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


def bench_step(iters=100, reps=3):
    torch.backends.cudnn.allow_tf32 = True
    notes, note = [], ops.note_library_path
    ops.note_library_path = lambda key, message: notes.append(message) if key == "conv_backward_aten" else None
    arms = {"kernels_tf32": qat_step("tf32")}
    ops.note_library_path = note
    arms["stock_cudnn"] = qat_step("cudnn")
    ms = {k: [] for k in arms}
    for _ in range(reps):
        for k, arm in arms.items():                       # alternately, in one process
            ms[k].append(replay_ms(arm[0], iters))
    out = {k: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v), "runs_ms": v}
           for k, v in ms.items()}
    out["speedup_stock_over_kernels"] = out["stock_cudnn"]["median_ms"] / out["kernels_tf32"]["median_ms"]
    out["kernels_tf32_conv_backward_on_aten"] = sorted(set(notes))     # layers left on cuDNN, from the captured step
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r04_pw_wgrad_bench.json")
    ap.add_argument("--iters", type=int, default=100)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pw_wgrad.py measures on a CUDA device; none is visible")
    res = {"card": card(), "layers_l2_state": "operands L2-resident: the same x, g and gw in every call",
           "layers": bench_layers(), "qat_step_mobilenetv2_po2plus_4bit_b128": bench_step(a.iters)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["qat_step_mobilenetv2_po2plus_4bit_b128"], indent=1))


if __name__ == "__main__":
    main()
