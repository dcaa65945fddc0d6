"""PTQ inference forward of bf16 models (BASELINE.json configs 0, 2 and 3: ResNet-20 4-bit, MobileNetV2 4-bit,
MobileViT-xs 8-bit at 224x224; PO2+ by default, or --quantizer lin / lin+ on the same models): the model cast to bf16,
then quantize_model, eval mode, eval-mode norms folded (fold_conv_bn), each forward captured in a CUDA graph.  Times our
kernels (bf16 activations) against the same bf16 model with its convs on cuDNN, and for reference the fp32 model on our
kernels (tf32 mode); the three graphs replay in alternation within one process, several rounds, so that clocks and
neighbours affect each alike.  For lin / lin+ each row also times quantize_model itself on the bf16 model: the bf16 lin
kernel against the op-by-op ATen form (PO2_LIN=aten), alternating.  The card's name and power limit are read in the
same run.

    python tools/bench_bf16_inference.py [--quantizer po2+] [--out profiles/r05_bf16_inference.json] [--rounds 5]
                                         [--iters 20]
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import po2_quantization_b200 as P  # noqa: E402
from po2_quantization_b200 import ops  # noqa: E402
from workloads import mobilenet_v2_cifar, mobilevit_xs, resnet_cifar  # noqa: E402

CASES = [
    ("config 0: resnet20 {q} 4b PTQ, B=128, 32x32", lambda: resnet_cifar(20, 10, None, 4), 4, 128, (32, 32)),
    ("config 2: mobilenetv2 {q} 4b PTQ, B=128, 32x32", lambda: mobilenet_v2_cifar(10, None, 4), 4, 128, (32, 32)),
    ("config 3: mobilevit-xs {q} 8b PTQ, B=256, 224x224", lambda: mobilevit_xs((224, 224), 1000, (1, 1), None, 8), 8, 256,
     (224, 224)),
]


def capture(fn):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s), torch.no_grad():
        for _ in range(3):
            fn()
        torch.cuda.current_stream().synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            out = fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    return g, out


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


def build(make, bits, dtype, quantizer):
    torch.manual_seed(8)
    m = make().cuda().to(dtype).eval()              # cast first: quantize_model tags the parameters it writes
    P.quantize_model(m, quantizer, bits)
    P.fold_conv_bn(m)
    return m


def quantize_model_ms(make, bits, quantizer, rounds):
    """host clock around quantize_model of the bf16 model (ending in a device synchronise), the bf16 lin kernel against
    the op-by-op ATen form (PO2_LIN=aten), alternating; a fresh copy of the same weights each time"""
    torch.manual_seed(8)
    m0 = make().cuda().to(torch.bfloat16).eval()
    times = {"kernel": [], "aten": []}
    old = os.environ.get("PO2_LIN")
    try:
        for r in range(rounds + 1):                  # round 0 warms up both paths
            for key, env in (("kernel", "cuda"), ("aten", "aten")):
                m = copy.deepcopy(m0)
                os.environ["PO2_LIN"] = env
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                P.quantize_model(m, quantizer, bits)
                torch.cuda.synchronize()
                if r:
                    times[key].append((time.perf_counter() - t0) * 1e3)
    finally:
        if old is None:
            os.environ.pop("PO2_LIN", None)
        else:
            os.environ["PO2_LIN"] = old
    return times


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quantizer", choices=("po2+", "lin", "lin+"), default="po2+")
    ap.add_argument("--out", default="profiles/r05_bf16_inference.json")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    quantizer = P.quantizer_dict[a.quantizer]
    lin = a.quantizer in ("lin", "lin+")
    rows = []
    for name, make, bits, B, img in CASES:
        name = name.format(q=a.quantizer)
        torch.manual_seed(9)
        x = torch.randn(B, 3, *img, device="cuda")
        mb, mf = build(make, bits, torch.bfloat16, quantizer), build(make, bits, torch.float32, quantizer)
        xb = x.to(torch.bfloat16)
        graphs, outs = {}, {}
        for key, mode, m, inp in (("po2_bf16", "tf32", mb, xb), ("cudnn_bf16", "cudnn", mb, xb),
                                  ("po2_fp32_tf32", "tf32", mf, x)):
            ops.set_conv_mode(mode)
            graphs[key], outs[key] = capture(lambda m=m, inp=inp: m(inp))
        ops.set_conv_mode(ops.DEFAULT_CONV_MODE)
        n0 = ops.LAUNCHES
        with torch.no_grad():
            mb(xb)
        po2_launches = ops.LAUNCHES - n0
        times = {k: [] for k in graphs}
        for _ in range(a.rounds):
            for k, g in graphs.items():
                times[k].append(replay_ms(g, a.iters))
        ref = outs["cudnn_bf16"].float()
        rel = ((outs["po2_bf16"].float() - ref).abs().max() / ref.abs().max()).item()
        row = {"case": name, "batch": B, "po2_library_launches_per_forward": po2_launches,
               "ms": {k: sorted(v) for k, v in times.items()},
               "median_ms": {k: sorted(v)[len(v) // 2] for k, v in times.items()},
               "logits_max_rel_diff_po2_vs_cudnn_bf16": rel}
        med = row["median_ms"]
        row["speedup_po2_bf16_vs_cudnn_bf16"] = med["cudnn_bf16"] / med["po2_bf16"]
        row["speedup_po2_bf16_vs_po2_fp32_tf32"] = med["po2_fp32_tf32"] / med["po2_bf16"]
        if lin:
            qt = quantize_model_ms(make, bits, quantizer, a.rounds)
            row["quantize_model_bf16_ms"] = {k: sorted(v) for k, v in qt.items()}
            row["quantize_model_bf16_median_ms"] = {k: sorted(v)[len(v) // 2] for k, v in qt.items()}
        rows.append(row)
        print(json.dumps(row), flush=True)
        del graphs, outs, mb, mf
        torch.cuda.empty_cache()
    result = {"device": card(), "torch": torch.__version__, "quantizer": a.quantizer, "rounds": a.rounds,
              "iters_per_round": a.iters,
              "timing": "CUDA events around graph replays, median over rounds; the three graphs alternate per round",
              "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"device": result["device"]}))


if __name__ == "__main__":
    main()
