#!/usr/bin/env python
"""bench.py -- the reference's headline metric on B200: quantized-conv images/sec (ResNet-56 CIFAR-10,
PO2 4-bit QAT forward + STE backward + SGD, batch 128 per GPU) and quantizer GB/s vs HBM peak.

    python bench.py --gpus N --steps K --warmup W            # our arm (N>1 under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results as DIR/*.npy

One JSON line on rank 0.
  value      whole-job images/s of the QAT step with inputs resident in HBM (CUDA-graph replay)
  e2e        the same step fed from pinned host memory with the loss read back every step
  roofline   the dominant kernel of the timed step (the tcgen05 conv forward) timed live per layer
             class with CUDA events against MEASURED_PEAKS.json; `roofline_quantizer` is the same for
             the quantizer's streaming kernels
  cpu_baseline  the reference's step on this box's host cores (the unmodified reference files when
             baseline/_ref is staged -- kind "reference" -- else the oracle's op-for-op port)
At N=1 rank 0 also reports, under `extra` (none of it inside the timed region of `value`):
  step variants   tf32 operands; the reference's OWN models/resnet.py (stock nn.SyncBatchNorm + ReLU
                  around the drop-in QuantizedConv2d) -- what an unmodified checkout gets
  gpu_oracle      the reference's torch code on this GPU (stock ATen / cuDNN, TF32 default), eager and
                  CUDA-graph captured -- BASELINE.md section 3 (2), the same-box kernel to beat
  configs         BASELINE.json configs[0], [2], [3] (ResNet-20 PTQ, MobileNetV2, MobileViT 224 B=256)
  quantizer_sweep configs[4] compressed: 2^20..2^32 x {fp32, bf16} x bits {2,4,8} x {codes, no codes}
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "resnet56_cifar10_po2_4bit_qat_fwd_bwd_sgd"
METRIC = "quantized-conv images/sec (ResNet-56 PO2 4-bit QAT fwd+STE bwd); quantizer GB/s vs HBM peak in `roofline_quantizer`"
DATA = "synthetic (randn images 3x32x32, randint labels; kaiming-init weights, seed 8)"
CONFIG_KEYS = ("workload", "batch_per_gpu", "global_batch", "parallelism", "device", "cuda_graph", "l2", "conv_backend",
               "conv_operands", "norm_backend", "weight_quantization", "model_source", "top1_identity",
               "bn_exchange_timeouts", "last_loss")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "source": "fallback (B200_PROFILING.md)"}


def full_config(**kw):
    """both arms emit the same config keys (the driver compares them)"""
    return {k: kw.get(k) for k in CONFIG_KEYS}


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                f = [t.strip() for t in out.strip().split(",")]
                if len(f) >= 7:
                    self.rows.append(f)
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm = sorted(int(float(r[0])) for r in self.rows if r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------
# the QAT step (BASELINE.json configs[1])
# ------------------------------------------------------------------------------------------------
def build_training(device, world, local_rank, source="workload"):
    """source "workload": workloads/resnet_cifar.py (FusedSyncBatchNorm takes add + ReLU);
    "reference_files": the reference's own models/resnet.py, unmodified, on the drop-in classes."""
    import po2_quantization_b200 as P
    torch.manual_seed(8)
    if source == "reference_files":
        from workloads import reference_files as RF
        ns = RF.load("dropin")
        if ns is None:
            return None
        model = ns.get_model("resnet56", 10, P.PowerOfTwoQuantizer, 4, (32, 32)).to(device).train()
    elif source == "reference_files_fused_norm":
        # the reference's own models/resnet.py, unmodified, plus ONE added line in the training script:
        # po2_quantization_b200.fuse_batchnorm(model) -- its nn.SyncBatchNorm modules run on this library's norm kernels
        from workloads import reference_files as RF
        ns = RF.load("dropin")
        if ns is None:
            return None
        model = ns.get_model("resnet56", 10, P.PowerOfTwoQuantizer, 4, (32, 32)).to(device).train()
        P.fuse_batchnorm(model)
    elif source == "workload_stock_norm":
        from workloads import resnet_cifar
        model = resnet_cifar(56, 10, P.PowerOfTwoQuantizer, 4, norm_cls=nn.SyncBatchNorm).to(device).train()
    else:
        from workloads import resnet_cifar
        model = resnet_cifar(56, 10, P.PowerOfTwoQuantizer, 4).to(device).train()
    if os.environ.get("PO2_PREFETCH", "1") == "1":
        # quantize all 56 weights in ONE multi-tensor launch at the start of each forward instead of one
        # by one in front of each conv (po2_quantization_b200/prefetch.py); same arithmetic, same results
        P.enable_weight_prefetch(model)
    # weight-gradient kernels on a side stream, joined at the end of backward (ops.set_wgrad_overlap): safe here
    # because the step zeroes gradients to None and nothing hooks them; torch DDP's reducer hooks would read them
    P.ops.set_wgrad_overlap(os.environ.get("PO2_WGRAD_STREAM", "1") == "1" and os.environ.get("PO2_DDP", "0") != "1"
                            and os.environ.get("PO2_GRAD_OVERLAP", "0") != "1")
    if world > 1:
        if os.environ.get("PO2_DDP", "0") == "1":
            # torch's DistributedDataParallel, as the reference wraps its model (train.py:153-155)
            model = nn.parallel.DistributedDataParallel(model, device_ids=[local_rank], gradient_as_bucket_view=True,
                                                        broadcast_buffers=False)
        else:
            # same arithmetic, coalesced NCCL all-reduce(AVG) per bucket (distributed.BatchSharded)
            from po2_quantization_b200.distributed import BatchSharded
            model = BatchSharded(model, overlap=os.environ.get("PO2_GRAD_OVERLAP", "0") == "1",
                                 buckets=int(os.environ.get("PO2_GRAD_BUCKETS", "4")))
    # reference train.py:51-56: SGD momentum 0.9, wd 1e-4, lr 0.1 * world
    # po2_quantization_b200.optim.SGD: torch.optim.SGD whose step() is one launch per 96 tensors (same roundings)
    sgd = torch.optim.SGD if os.environ.get("PO2_SGD", "ours") == "torch" else P.optim.SGD
    opt = sgd(model.parameters(), lr=0.1 * world, momentum=0.9, weight_decay=1e-4)
    crit = nn.CrossEntropyLoss()
    return model, opt, crit


def _parallelism_note():
    from po2_quantization_b200 import batchnorm
    grads = ("torch DDP buckets" if os.environ.get("PO2_DDP", "0") == "1"
             else ("coalesced NCCL all-reduce(AVG) of the gradients in buckets, issued from grad hooks under backward"
                   if os.environ.get("PO2_GRAD_OVERLAP", "0") == "1"
                   else "one coalesced NCCL all-reduce(AVG) of all gradients behind backward"))
    ex = [e for e in batchnorm._exchanges.values()]
    mode = os.environ.get("PO2_BN_EXCHANGE", "peer")
    bn = ("SyncBatchNorm statistics exchanged inside the BN kernels over NVLink peer stores" if any(e is not None for e in ex)
          else "per-rank BatchNorm statistics" if mode == "local" else "SyncBatchNorm statistics over NCCL all_gather/all_reduce")
    return f" (batch-sharded; {grads}; {bn})"


def _exchange_timeouts():
    """number of peer mailboxes whose poll ever timed out (must be 0)"""
    from po2_quantization_b200 import batchnorm
    return sum(1 for e in batchnorm._exchanges.values() if e is not None and e.error_flag() != 0)


def activation_bytes_estimate(batch):
    # saved activations of ResNet-56 at 32x32: 19 layer-1 convs+bn+relu at 16ch/32^2, 18 at 32ch/16^2, 18 at 64ch/8^2
    per_img = (19 * 16 * 32 * 32 + 18 * 32 * 16 * 16 + 18 * 64 * 8 * 8) * 4 * 3
    return per_img * batch


def operand_label(mode):
    return {"tc": "bf16 operands (PO2 weights exact, activations/gradients rounded to bf16), f32 accumulate",
            "tf32": "tf32 operands (PO2 weights exact, activations keep 10 mantissa bits), f32 accumulate",
            "fp32": "f32 FMA", "cudnn": "cuDNN (TF32 by default)"}[mode]


class StepHarness:
    """One training configuration: model + optimiser + a CUDA graph of the whole step, on the current stream."""

    def __init__(self, a, world, rank, local_rank, device, source="workload"):
        from po2_quantization_b200 import ops
        self.ops, self.world, self.rank, self.device, self.a = ops, world, rank, device, a
        built = build_training(device, world, local_rank, source)
        self.ok = built is not None
        if not self.ok:
            return
        self.model, self.opt, self.crit = built
        B = a.batch
        g = torch.Generator().manual_seed(1000 + rank)
        self.x_host = torch.randn(B, 3, 32, 32, generator=g).pin_memory()
        self.y_host = torch.randint(0, 10, (B,), generator=g).pin_memory()
        self.x_dev = self.x_host.to(device)
        self.y_dev = self.y_host.to(device)
        self.loss_buf = torch.zeros((), device=device)
        self.graph = None
        self.launches_per_step = None

    def step(self):
        self.opt.zero_grad()  # reference train.py:81 (set_to_none=True: no fill / accumulate kernels)
        loss = self.crit(self.model(self.x_dev), self.y_dev)
        loss.backward()
        if hasattr(self.model, "average_gradients"):
            self.model.average_gradients()
        self.opt.step()
        self.loss_buf.copy_(loss.detach())

    def capture(self):
        """CUDA graph of the whole step.  With N>1 the NCCL all-reduce and the SyncBatchNorm exchanges are
        captured too; DDP needs its bucket rebuild (iteration 2) to have happened, hence the eager steps."""
        ops, world = self.ops, self.world
        for _ in range(3):
            self.step()
        torch.cuda.synchronize()
        if not self.a.no_graph:
            try:
                for _ in range(11 if world > 1 else 3):
                    self.step()
                torch.cuda.current_stream().synchronize()
                if world > 1:
                    torch.distributed.barrier()
                self.graph = torch.cuda.CUDAGraph()
                ops.LAUNCHES = 0
                with torch.cuda.graph(self.graph, stream=torch.cuda.current_stream()):
                    self.step()
                self.launches_per_step = ops.LAUNCHES
                torch.cuda.synchronize()
            except Exception as e:  # pragma: no cover
                print(f"[bench] CUDA graph capture failed ({type(e).__name__}: {e}); running eagerly", file=sys.stderr)
                self.graph = None
        if self.launches_per_step is None:
            ops.LAUNCHES = 0
            self.step()
            self.launches_per_step = ops.LAUNCHES
        self.run = self.graph.replay if self.graph is not None else self.step

    def barrier(self):
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        if self.world > 1:
            t = torch.tensor([ms], device=self.device, dtype=torch.float64)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            return float(t.item())
        return ms

    def time_resident(self, steps, warmup):
        for _ in range(max(warmup, 3)):
            self.run()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            self.run()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1))

    def time_e2e(self, steps):
        """pinned host -> device copy of the batch every step, loss read back every step"""
        for _ in range(2):
            self.x_dev.copy_(self.x_host, non_blocking=True); self.y_dev.copy_(self.y_host, non_blocking=True)
            self.run(); self.loss_buf.item()
        self.barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        last = 0.0
        for _ in range(steps):
            self.x_dev.copy_(self.x_host, non_blocking=True)
            self.y_dev.copy_(self.y_host, non_blocking=True)
            self.run()
            last = self.loss_buf.item()            # device -> host read of the step's result
        f1.record()
        self.barrier()
        return self.max_over_ranks(f0.elapsed_time(f1)), last

    def weight_checksum(self):
        """sum of all parameters in fp64: identical on every rank iff the replicas stayed in lock-step"""
        with torch.no_grad():
            return float(sum(p.double().sum() for p in self.model.parameters()).item())

    def close(self):
        self.graph = None
        self.model = self.opt = None
        gc.collect()
        torch.cuda.empty_cache()


DUMP_LIMIT_BYTES = 64 * 2 ** 20


def step_outputs(model, loss_buf):
    """What a training step leaves its caller: the loss of the last step, the parameters after its SGD update and
    the norms' running statistics (floating-point tensors only; the integer batch counters are left out)."""
    out = {"loss": loss_buf.detach().float().cpu().numpy()}
    with torch.no_grad():
        for name, t in list(model.named_parameters()) + list(model.named_buffers()):
            if t.is_floating_point():
                out[name] = t.detach().float().cpu().numpy()
    return out


def dump_outputs(arrays, directory):
    """Write each array as <directory>/<name>.npy (float32), so that two builds run with the same arguments
    (hence the same seeded inputs) can be compared output for output."""
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: outputs of {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte dump limit")
    os.makedirs(directory, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), v)


def run_ours(a):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    from po2_quantization_b200 import ops

    # Everything (model/DDP construction, warm-up, capture, replay, timing events) runs on ONE side
    # stream: CUDA-graph capture is illegal on the legacy default stream, and DDP's AccumulateGrad
    # hooks must be created on the stream the captured step later runs on.
    # high priority: where the step forks (weight gradients on ops' side stream) the main branch's CTAs go first
    side = torch.cuda.Stream(device, priority=int(os.environ.get("PO2_MAIN_PRIORITY", "-1")))
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        _run_ours_on_stream(a, ops, world, rank, local_rank, device)
    if world > 1:
        # A captured graph keeps NCCL work objects alive and destroy_process_group() can then wait
        # forever at interpreter exit; every rank is past its last collective here, so leave hard.
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def _run_ours_on_stream(a, ops, world, rank, local_rank, device):
    B = a.batch
    parts = set(a.parts.split(","))
    h = StepHarness(a, world, rank, local_rank, device)

    if a.torch_profile:
        # kernel-time table of eager steps from torch.profiler (works under torchrun, where ncu does not):
        # rank 0 writes the per-kernel totals of 5 steps to the given path
        from torch.profiler import ProfilerActivity, profile
        for _ in range(12):
            h.step()
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                h.step()
            torch.cuda.synchronize()
        if rank == 0:
            rows = [(e.key, e.count, e.device_time_total) for e in prof.key_averages() if e.device_time_total > 0]
            rows.sort(key=lambda r: -r[2])
            tot = sum(r[2] for r in rows)
            with open(a.torch_profile, "w") as f:
                f.write(f"# 5 eager steps, world={world}; total device time {tot / 5:.1f} us per step\n")
                for k, c, t in rows:
                    f.write(f"{t / 5:10.1f} us/step {c // 5:5d} x  {100 * t / tot:5.1f}%  {k[:110]}\n")
            print(json.dumps({"torch_profile": a.torch_profile, "device_us_per_step": tot / 5}))
        return

    if a.graph_timeline:
        # device timeline of graph replays from torch.profiler (CUPTI): per-stream busy time, idle gaps on the
        # main branch, per-kernel totals inside the captured step (where the side branch overlaps the main one)
        from torch.profiler import ProfilerActivity, profile
        h.capture()
        for _ in range(5):
            h.run()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                h.run()
            torch.cuda.synchronize()
        if rank == 0:
            evs = [e for e in prof.events() if e.device_type.name == "CUDA" and e.time_range.end > e.time_range.start]
            evs.sort(key=lambda e: e.time_range.start)
            rows = [{"name": e.name[:90], "t0": e.time_range.start, "t1": e.time_range.end} for e in evs]
            t_first, t_last = rows[0]["t0"], max(r["t1"] for r in rows)
            # union of busy intervals
            busy, cur0, cur1 = 0.0, None, None
            for r in rows:
                if cur1 is None or r["t0"] > cur1:
                    if cur1 is not None:
                        busy += cur1 - cur0
                    cur0, cur1 = r["t0"], r["t1"]
                else:
                    cur1 = max(cur1, r["t1"])
            busy += cur1 - cur0
            per = {}
            for r in rows:
                k = r["name"].split("(")[0]
                d = per.setdefault(k, [0, 0.0])
                d[0] += 1
                d[1] += r["t1"] - r["t0"]
            top = sorted(per.items(), key=lambda kv: -kv[1][1])
            with open(a.graph_timeline, "w") as f:
                f.write(f"# 3 graph replays, world={world}: span {(t_last - t_first) / 3:.1f} us/step, device busy (union) "
                        f"{busy / 3:.1f} us/step, sum of kernel durations {sum(v[1] for v in per.values()) / 3:.1f} us/step\n")
                for k, (c, t) in top:
                    f.write(f"{t / 3:10.1f} us/step {c // 3:5d} x {t / c:8.2f} us each  {k}\n")
                f.write("# timeline of the second replay (start us, duration us, name)\n")
                n = len(rows) // 3
                base = rows[n]["t0"]
                for r in rows[n:2 * n]:
                    f.write(f"{r['t0'] - base:10.2f} {r['t1'] - r['t0']:8.2f} {r['name']}\n")
            print(json.dumps({"graph_timeline": a.graph_timeline, "span_us_per_step": (t_last - t_first) / 3,
                              "busy_us_per_step": busy / 3}))
        return

    if a.profile_step:
        # one eager step between cudaProfilerStart/Stop: `ncu --profile-from-start off` lists exactly
        # the kernels of a step (profiles/ launch list)
        for _ in range(3):
            h.step()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStart()
        h.step()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
        print(json.dumps({"profile_step": True, "launches_of_libpo2b200": ops.LAUNCHES}))
        return

    h.capture()
    with ClockSampler(local_rank) as clk:
        ms_total = h.time_resident(a.steps, a.warmup)
        ms_e2e, last = h.time_e2e(a.steps)
    clocks = clk.summary()
    checksum = h.weight_checksum()
    if world > 1:
        # replicas must hold bit-identical weights after the timed steps (gradient averaging + SyncBatchNorm
        # exchange correct on every rank): compare the fp64 checksums
        t = torch.tensor([checksum, -checksum], device=device, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        replicas_identical = bool(t[0].item() == -t[1].item())
        torch.distributed.barrier()
    else:
        replicas_identical = True
    timeouts = _exchange_timeouts()
    if rank != 0:
        return
    outputs = step_outputs(h.model, h.loss_buf) if a.dump_outputs else None
    mode = ops.get_conv_mode()
    ms_step = ms_total / a.steps
    out = {
        "metric": METRIC, "value": world * B * a.steps / (ms_total / 1e3), "unit": "images/s",
        "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": operand_label(mode),
        "data": DATA,
        "config": full_config(
            workload=WORKLOAD, batch_per_gpu=B, global_batch=B * world, device="cuda",
            parallelism=f"dp{world}" + (_parallelism_note() if world > 1 else ""),
            cuda_graph=h.graph is not None,
            l2="working set per step ~%d MB of saved activations > 126 MB L2; no flush needed" % (activation_bytes_estimate(B) // 2 ** 20),
            conv_backend=ops.conv_backend_name(), conv_operands=operand_label(mode), last_loss=last,
            norm_backend="po2 FusedSyncBatchNorm kernels (norm + residual add + ReLU, forward and backward)",
            weight_quantization=("one multi-tensor launch per step (prefetch)" if os.environ.get("PO2_PREFETCH", "1") == "1"
                                 else "one launch per layer"),
            model_source="workloads/resnet_cifar.py (layer graph of models/resnet.py; FusedSyncBatchNorm); the reference's "
                         "own models/resnet.py, unmodified, is timed in extra.step_variants.reference_model_files (torch norms) and "
                         "reference_model_files_plus_fuse_batchnorm (one added line: po2_quantization_b200.fuse_batchnorm(model))",
            top1_identity="asserted bit-for-bit in fp32-accumulate mode; bf16/tf32 operand modes are checked on decisive "
                          "margins (tests/test_conv_gpu.py::test_ptq_quantize_model_and_forward_resnet20_top1)",
            bn_exchange_timeouts=timeouts),
        "e2e": {"value": world * B * a.steps / (ms_e2e / 1e3), "unit": "images/s",
                "h2d_bytes_per_step": h.x_host.numel() * 4 + h.y_host.numel() * 8, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / a.steps},
        "gpu_launches": h.launches_per_step * a.steps,
        "gpu_launches_per_step": h.launches_per_step,
        "clocks": clocks,
        "weights_fp64_checksum": checksum, "replicas_identical_after_timed_steps": replicas_identical,
    }
    h.close()
    if world == 1:
        out["roofline"] = conv_forward_roofline(device, B) if "roofline" in parts else None
        qroof, qrows = quantizer_roofline(device, a) if "roofline" in parts else (None, None)
        out["roofline_quantizer"], out["roofline_quantizer_rows"] = qroof, qrows
        extra = {}
        if "variants" in parts:
            extra["step_variants"] = step_variants(a, device, ms_step)
        if "oracle" in parts:
            extra["gpu_oracle"] = gpu_oracle_step(a, device, ms_step)
        if "configs" in parts:
            extra["configs"] = other_configs(device)
        if "sweep" in parts:
            extra["quantizer_sweep"] = quantizer_sweep(device, a.sweep_max_log2)
        out["extra"] = extra
        if not a.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(B, steps=2)
    print(json.dumps(out), flush=True)
    if outputs is not None:
        dump_outputs(outputs, a.dump_outputs)


# ------------------------------------------------------------------------------------------------
# step variants and the GPU oracle (N=1, outside the timed region of `value`)
# ------------------------------------------------------------------------------------------------
def step_variants(a, device, ms_main):
    """The same QAT step (a) with tf32 operands, (b) on the reference's own models/resnet.py -- stock
    nn.SyncBatchNorm + nn.ReLU modules around the drop-in QuantizedConv2d, which is what an unmodified
    checkout of the reference gets from this library."""
    from po2_quantization_b200 import ops
    res = {"main_ms": ms_main}
    prev = ops.get_conv_mode()
    other = "tc" if prev == "tf32" else "tf32"
    for name, mode, source in ((("bf16_operands" if other == "tc" else "tf32_operands"), other, "workload"),
                               ("reference_model_files", prev, "reference_files"),
                               ("reference_model_files_plus_fuse_batchnorm", prev, "reference_files_fused_norm"),
                               ("reference_model_files_" + ("bf16" if other == "tc" else "tf32"), other, "reference_files")):
        try:
            ops.set_conv_mode(mode)
            h = StepHarness(a, 1, 0, device.index or 0, device, source)
            if not h.ok:
                h = StepHarness(a, 1, 0, device.index or 0, device, "workload_stock_norm")
                src = "workloads/resnet_cifar.py with stock nn.SyncBatchNorm (baseline/_ref not staged)"
            else:
                src = {"reference_files": "models/resnet.py of the reference, unmodified (baseline/_ref)",
                       "reference_files_fused_norm": "models/resnet.py of the reference, unmodified (baseline/_ref), plus one "
                       "line in the training script: po2_quantization_b200.fuse_batchnorm(model)"}.get(source, "workloads/resnet_cifar.py")
            h.capture()
            ms = h.time_resident(min(a.steps, 10), 3) / min(a.steps, 10)
            res[name] = {"ms_per_step": ms, "images_per_s": a.batch / ms * 1e3, "conv_operands": operand_label(mode),
                         "model": src, "cuda_graph": h.graph is not None, "launches_per_step": h.launches_per_step,
                         "last_loss": float(h.loss_buf.item())}
            h.close()
        except Exception as e:  # pragma: no cover
            res[name] = {"error": f"{type(e).__name__}: {e}"}
        finally:
            ops.set_conv_mode(prev)
    return res


def _reference_training_step(device, batch, seed_rank=0):
    """The reference's own training step (train.py:79-92) on `device`: the unmodified reference files when
    staged (kind "reference"), else the oracle's op-for-op torch restatement (kind "port")."""
    from workloads import reference_files as RF
    ns = RF.load("stock")
    torch.manual_seed(8)
    if ns is not None:
        model = ns.get_model("resnet56", 10, ns.quantizers.PowerOfTwoQuantizer, 4, (32, 32))
        kind, what = "reference", "unmodified reference files (baseline/_ref: models/resnet.py, utils/quantizers.py)"
    else:
        from oracle.po2_oracle_torch import PO2, QuantizedConv2dOracle
        from workloads import resnet_cifar
        model = resnet_cifar(56, 10, PO2, 4, conv_cls=QuantizedConv2dOracle)
        kind, what = "port", "oracle/po2_oracle_torch.py (stock ATen ops == what the reference runs)"
    model = model.to(device).train()
    opt = torch.optim.SGD(model.parameters(), lr=0.1, momentum=0.9, weight_decay=1e-4)
    crit = nn.CrossEntropyLoss()
    g = torch.Generator().manual_seed(1000 + seed_rank)
    x = torch.randn(batch, 3, 32, 32, generator=g).to(device)
    y = torch.randint(0, 10, (batch,), generator=g).to(device)
    loss_buf = torch.zeros((), device=device)

    def step():
        opt.zero_grad()  # reference train.py:81
        loss = crit(model(x), y)
        loss.backward()
        opt.step()
        loss_buf.copy_(loss.detach())
    return step, loss_buf, kind, what, model


def _time_loop(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def gpu_oracle_step(a, device, ms_main):
    """BASELINE.md section 3 (2): the reference's torch code on THIS GPU -- stock ATen elementwise
    quantizer ops, cuDNN convolutions (allow_tf32 at torch's default, True), stock BatchNorm -- eager (how
    train.py runs it) and CUDA-graph captured (launch overhead removed: the strongest same-box baseline)."""
    try:
        step, loss_buf, kind, what, _ = _reference_training_step(device, a.batch)
        for _ in range(5):
            step()
        iters = min(a.steps, 10)
        eager = _time_loop(step, iters)
        graph_ms = None
        try:
            torch.cuda.current_stream().synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=torch.cuda.current_stream()):
                step()
            for _ in range(3):
                g.replay()
            graph_ms = _time_loop(g.replay, iters)
        except Exception as e:  # pragma: no cover
            print(f"[bench] gpu_oracle graph capture failed: {type(e).__name__}: {e}", file=sys.stderr)
        res = {"kind": kind, "what": what, "device": torch.cuda.get_device_name(device),
               "cudnn_allow_tf32": bool(torch.backends.cudnn.allow_tf32), "eager_ms_per_step": eager,
               "eager_images_per_s": a.batch / eager * 1e3, "graph_ms_per_step": graph_ms,
               "graph_images_per_s": (a.batch / graph_ms * 1e3) if graph_ms else None,
               "ours_ms_per_step": ms_main, "speedup_vs_eager": eager / ms_main,
               "speedup_vs_graph": (graph_ms / ms_main) if graph_ms else None, "last_loss": float(loss_buf.item())}
        del g, step
        gc.collect()
        torch.cuda.empty_cache()
        return res
    except Exception as e:  # pragma: no cover
        return {"error": f"{type(e).__name__}: {e}"}


# ------------------------------------------------------------------------------------------------
# BASELINE.json configs[0], [2], [3]: inference forward, ours vs the reference's torch code on this GPU
# ------------------------------------------------------------------------------------------------
def _graph_forward_ms(model, x, iters=10):
    with torch.no_grad():
        for _ in range(3):
            model(x)
        torch.cuda.current_stream().synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=torch.cuda.current_stream()):
            out = model(x)
        for _ in range(2):
            g.replay()
        ms = _time_loop(g.replay, iters)
    top1 = out.argmax(1).clone()
    del g
    return ms, top1, out


def other_configs(device):
    import po2_quantization_b200 as P
    from po2_quantization_b200 import ops
    from workloads import mobilenet_v2_cifar, mobilevit_xs, reference_files as RF, resnet_cifar
    stock, dropin = RF.load("stock"), RF.load("dropin")
    rows = {}

    def oracle_model(name, bits, img, classes):
        if stock is None:
            return None
        torch.manual_seed(8)
        if name == "mobilevit224":
            m = RF.mobilevit_224(stock, classes, None, bits)
        else:
            m = stock.get_model(name, classes, None, bits, img)
        return m

    cases = [
        # (key, BASELINE config, ours builder, reference-file name, bits, batch, image, classes, flop per batch of quantized convs)
        ("config0_resnet20_po2plus_4b_ptq_fwd_b128", lambda: resnet_cifar(20, 10, None, 4), "resnet20", 4, 128, (32, 32), 10, 10.34e9),
        ("config2_mobilenetv2_po2plus_4b_ptq_fwd_b128", lambda: mobilenet_v2_cifar(10, None, 4), "mobilenet", 4, 128, (32, 32), 10, 1.40e9),
        ("config3_mobilevit_xs_224_patch1_po2plus_8b_ptq_fwd_b256", lambda: mobilevit_xs((224, 224), 1000, (1, 1), None, 8),
         "mobilevit224", 8, 256, (224, 224), 1000, 234.4e9),
    ]
    for key, build, refname, bits, B, img, classes, flop in cases:
        r = {"batch": B, "image": list(img), "bits": bits, "qconv_flop_per_batch": flop}
        try:
            torch.manual_seed(8)
            ref = oracle_model(refname, bits, img, classes)
            torch.manual_seed(8)
            m = build()
            if ref is not None:
                m.load_state_dict(ref.state_dict(), strict=True)       # same weights in all arms
            m = m.to(device).eval()
            mse = P.quantize_model(m, P.PowerOfTwoPlusQuantizer, bits)
            # inference: eval-mode norms (+ residual add, + activation) folded into the conv epilogues
            r["folded_conv_bn_pairs"] = P.fold_conv_bn(m)
            x = torch.randn(B, 3, *img, generator=torch.Generator().manual_seed(0)).to(device)
            ops.LAUNCHES = 0
            ms, top1, out = _graph_forward_ms(m, x)
            r.update({"ours_ms": ms, "ours_images_per_s": B / ms * 1e3, "ptq_mse": mse, "ours_launches_per_forward": ops.LAUNCHES // 4,
                      "ours_qconv_TFLOPs_if_all_time_were_conv": flop / ms / 1e9})
            # the same model object with its convs on cuDNN (isolates the conv kernels from the fused norms)
            ops.set_conv_mode("cudnn")
            try:
                ms_c, _, _ = _graph_forward_ms(m, x)
            finally:
                ops.set_conv_mode(ops.DEFAULT_CONV_MODE)
            r.update({"ours_with_cudnn_convs_ms": ms_c, "speedup_vs_own_cudnn_convs": ms_c / ms})
            if dropin is not None and refname != "mobilevit224":
                # the reference's own model file on the drop-in classes (stock norms/activations)
                torch.manual_seed(8)
                md = dropin.get_model(refname, classes, None, bits, img)
                md.load_state_dict(ref.state_dict(), strict=True)
                md = md.to(device).eval()
                P.quantize_model(md, P.PowerOfTwoPlusQuantizer, bits)
                ms_d, top1_d, _ = _graph_forward_ms(md, x)
                r.update({"reference_model_file_on_dropin_ms": ms_d, "reference_model_file_on_dropin_images_per_s": B / ms_d * 1e3})
                # ... plus two added lines in the evaluation script: fuse_batchnorm(model); fold_conv_bn(model)
                P.fuse_batchnorm(md)
                P.fold_conv_bn(md)
                ms_f, top1_f, _ = _graph_forward_ms(md, x)
                r.update({"reference_model_file_on_dropin_plus_fuse_and_fold_ms": ms_f,
                          "reference_model_file_plus_fuse_and_fold_top1_agreement": float((top1_f == top1_d).float().mean().item())})
                del md
            if ref is not None:
                ref = ref.to(device).eval()
                stock.quantizers.quantize_model(ref, stock.quantizers.PowerOfTwoPlusQuantizer, bits)
                with torch.no_grad():
                    for _ in range(3):
                        ref(x)
                    eager = _time_loop(lambda: ref(x), 5)
                ms_o, top1_o, out_o = _graph_forward_ms(ref, x)
                rel = ((out.double() - out_o.double()).abs().max() / out_o.double().abs().max()).item()
                r.update({"gpu_oracle_eager_ms": eager, "gpu_oracle_graph_ms": ms_o, "gpu_oracle_images_per_s": B / ms_o * 1e3,
                          "speedup_vs_gpu_oracle_graph": ms_o / ms, "speedup_vs_gpu_oracle_eager": eager / ms,
                          "logits_rel_err_vs_gpu_oracle": rel,
                          "top1_agreement_vs_gpu_oracle": float((top1 == top1_o).float().mean().item())})
            if key.startswith("config2"):
                # QAT-eval mode (test.py:133-159): the model keeps its quantizer and re-quantizes every forward
                torch.manual_seed(8)
                mq = mobilenet_v2_cifar(10, P.PowerOfTwoPlusQuantizer, 4).to(device).eval()
                P.enable_weight_prefetch(mq)
                ms_q, _, _ = _graph_forward_ms(mq, x)
                r.update({"ours_qat_eval_ms": ms_q, "ours_qat_eval_images_per_s": B / ms_q * 1e3})
                del mq
            del m, ref, x, out
        except Exception as e:  # pragma: no cover
            r["error"] = f"{type(e).__name__}: {e}"
        gc.collect()
        torch.cuda.empty_cache()
        rows[key] = r
    return rows


# ------------------------------------------------------------------------------------------------
# quantizer: roofline at one size + the compressed sweep of BASELINE.json configs[4]
# ------------------------------------------------------------------------------------------------
def _timed_each(fn, iters=10, flush=None):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for p, q in ev:
        if flush is not None:
            flush.add_(1)
        p.record(); fn(); q.record()
    torch.cuda.synchronize()
    ts = sorted(p.elapsed_time(q) for p, q in ev)
    return sum(ts) / len(ts), ts[len(ts) // 2]


def quantizer_roofline(device, a):
    """Quantizer streaming kernels at 2^log2n elements, timed one launch at a time with CUDA events
    on the launching stream.  Algorithmic bytes (SURVEY.md 8d): absmax reads es, quantize reads es
    and writes es per element."""
    from po2_quantization_b200 import ops
    pk = peaks()
    res = []
    for dt, es, name in ((torch.float32, 4, "f32"), (torch.bfloat16, 2, "bf16")):
        n = 1 << a.sweep_log2
        x = torch.randn(n, device=device, dtype=torch.float32).to(dt)
        y = torch.empty_like(x)
        s = torch.empty((), dtype=torch.float32, device=device)
        t_abs, _ = _timed_each(lambda: ops.absmax_out(x, s))
        t_q, _ = _timed_each(lambda: ops.quantize_out(x, y, s, 4, 1, False))
        t_all, _ = _timed_each(lambda: ops.quantize_fused_out(x, y, s, 4, 1, False))
        res.append({"kernel": f"po2::quantize_kernel<{name}> (pass 2 of po2_quantize_fused)", "dtype": name,
                    "elements": n, "bytes_per_element": 2 * es, "ms": t_q,
                    "achieved": 2 * es * n / t_q / 1e6, "absmax_ms": t_abs,
                    "absmax_GBs": es * n / t_abs / 1e6, "both_passes_ms": t_all,
                    "both_passes_GBs": 3 * es * n / t_all / 1e6})
        del x, y
    r0 = res[0]
    roof = {"bound": "hbm", "kernel": r0["kernel"], "achieved": r0["achieved"], "peak": pk["hbm_gbs"],
            "unit": "GB/s", "frac": r0["achieved"] / pk["hbm_gbs"],
            # dram__bytes_read.sum + dram__bytes_write.sum of this kernel at this size from the committed
            # `ncu --set full` captures (profiles/r01_ncu_quantize_kernel_f32_2p28.csv: 1.074 + 1.028 GB;
            # profiles/r01_ncu_quantize_kernel_f32_2p30.csv: 4.295 + 4.248 GB)
            "traffic": {28: 2.102e9, 30: 8.543e9}.get(a.sweep_log2), "algorithmic_bytes": 8.0 * (1 << a.sweep_log2),
            "peak_source": pk["source"], "frac_of_nominal_8TBs": r0["achieved"] / 8000.0,
            "note": "algorithmic bytes = 8 B/element (4 read + 4 written) x 2^%d fp32 elements per launch; "
                    "inputs (%.1f GB) larger than L2" % (a.sweep_log2, 4 * (1 << a.sweep_log2) / 1e9)}
    for r in res:
        r["frac_quantize_pass"] = r["achieved"] / pk["hbm_gbs"]
        r["frac_both_passes"] = r["both_passes_GBs"] / pk["hbm_gbs"]
        r["frac_absmax_pass"] = r["absmax_GBs"] / pk["hbm_gbs"]
    torch.cuda.empty_cache()
    return roof, res


def quantizer_sweep(device, max_log2=32):
    """BASELINE.json configs[4], compressed: N = 2^20, 2^22, ..., 2^max_log2; fp32 and bf16; bits 2, 4, 8;
    with and without packed codes; po2 everywhere plus po2+ at 4 bits.  What `Q.forward` costs (both
    passes): algorithmic bytes = 3*es (+ bits/8 with codes, rounded up to the packed byte) per element.
    L2 is flushed between iterations while the tensors are smaller than 256 MB."""
    from po2_quantization_b200 import ops
    pk = peaks()
    flush_buf = torch.zeros(320 * 1024 * 1024 // 4, dtype=torch.int32, device=device)
    rows = []
    for dt, es, name in ((torch.float32, 4, "f32"), (torch.bfloat16, 2, "bf16")):
        for lg in range(20, max_log2 + 1, 2):
            n = 1 << lg
            try:
                chunk = min(n, 1 << 28)
                x = torch.empty(n, device=device, dtype=dt)
                gen = torch.Generator(device=device).manual_seed(1234)
                for i in range(0, n, chunk):            # randn in chunks: no 2x fp32 temporary for the 16 GiB case
                    x[i:i + chunk] = torch.randn(chunk, device=device, dtype=torch.float32, generator=gen).to(dt)
                y = torch.empty_like(x)
                s = torch.empty((), dtype=torch.float32, device=device)
                codes = torch.empty(n, dtype=torch.uint8, device=device)
                flush = flush_buf if n * es < 256 * 1024 * 1024 else None
                iters = 10 if lg <= 28 else 5
                for bits, plus in ((2, False), (4, False), (4, True), (8, False)):
                    mean, med = _timed_each(lambda: ops.quantize_fused_out(x, y, s, bits, 1, plus), iters, flush)
                    cb = 0.5 if bits <= 4 else 1.0
                    mean_c, med_c = _timed_each(lambda: ops.quantize_fused_out(x, y, s, bits, 1, plus, codes=codes[:int(n * cb)]),
                                                iters, flush)
                    rows.append({"dtype": name, "log2n": lg, "bits": bits, "quantizer": "po2+" if plus else "po2",
                                 "ms": med, "GBs": 3 * es * n / med / 1e6, "frac": 3 * es * n / med / 1e6 / pk["hbm_gbs"],
                                 "ms_codes": med_c, "GBs_codes": (3 * es + cb) * n / med_c / 1e6,
                                 "frac_codes": (3 * es + cb) * n / med_c / 1e6 / pk["hbm_gbs"]})
                del x, y, codes
            except torch.cuda.OutOfMemoryError:  # pragma: no cover
                rows.append({"dtype": name, "log2n": lg, "error": "out of memory"})
            torch.cuda.empty_cache()
    big = [r for r in rows if "frac" in r and r["log2n"] >= 28]
    return {"peak_GBs": pk["hbm_gbs"], "peak_source": pk["source"], "bytes_per_element": "3*es (+0.5 or 1 with codes)",
            "min_frac_at_2p28_and_up": min((r["frac"] for r in big), default=None),
            "min_frac_codes_at_2p28_and_up": min((r["frac_codes"] for r in big), default=None), "rows": rows}


# ------------------------------------------------------------------------------------------------
# the dominant kernel of the step: tcgen05 conv forward, per ResNet-56 layer class
# ------------------------------------------------------------------------------------------------
def conv_forward_roofline(device, batch):
    """Quantized-conv FORWARD of the ResNet-56 layer classes, timed live in CUDA graphs (the pack +
    conv kernels of one QuantizedConv2d.forward), with a cold L2 (a 320 MB buffer is rewritten before
    every conv).  These layers have 36-144 flop/B at the fp32 NCHW module boundary, so the binding
    roof is HBM: algorithmic bytes = 4*(B*C*H*W + B*K*P*Q)."""
    import torch.nn.functional as F
    from po2_quantization_b200 import _lib, ops
    pk = peaks()
    flush = torch.zeros(320 * 1024 * 1024 // 4, dtype=torch.int32, device=device)
    compute = ops.COMPUTE.get(ops.get_conv_mode(), 0)

    def graph_ms(body, reps=10, iters=5):
        body()
        torch.cuda.current_stream().synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=torch.cuda.current_stream()):
            for _ in range(reps):
                body()
        torch.cuda.synchronize()
        g.replay()
        torch.cuda.synchronize()
        ts = []
        for _ in range(iters):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); g.replay(); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return sorted(ts)[len(ts) // 2] / reps

    t_flush = graph_ms(lambda: flush.add_(1))
    layers = [("16->16 3x3 @32x32", 16, 32, 16, 18), ("32->32 3x3 @16x16", 32, 16, 32, 17), ("64->64 3x3 @8x8", 64, 8, 64, 17)]
    rows, tot_us, tot_cudnn, tot_flop, tot_bytes = [], 0.0, 0.0, 0.0, 0.0
    for name, C, HW, K, count in layers:
        x = torch.randn(batch, C, HW, HW, device=device)
        w = torch.randn(K, C, 3, 3, device=device) * 0.1
        y, _, scale, _, _ = torch.ops.po2.quantize_full(w, 4, 1, False)
        out = torch.empty(batch, K, HW, HW, device=device)

        # the launch the timed step performs: the conv kernel alone, its weight operand packed by the
        # step's multi-tensor quantizer launch (prefetch.py); `us_with_pack` = the un-prefetched QAT forward
        packed = ops.conv2d_pack(y, scale, x.shape, 1, 1, 1, compute)

        def ours():
            flush.add_(1)
            torch.ops.po2.conv2d_packed(x, packed, scale, K, 3, 3, 1, 1, 1, compute)

        def ours_with_pack():
            flush.add_(1)
            ops.conv2d_out(x, y, scale, out, 1, 1, 1, compute)

        def cudnn():
            flush.add_(1)
            F.conv2d(x, y, None, 1, 1)
        us = (graph_ms(ours) - t_flush) * 1e3
        us_p = (graph_ms(ours_with_pack) - t_flush) * 1e3
        us_c = (graph_ms(cudnn) - t_flush) * 1e3
        flop = 2.0 * batch * K * HW * HW * C * 9
        byts = 4.0 * (x.numel() + out.numel())
        kind = _lib.load().po2_conv2d_kernel_kind(batch, C, HW, HW, K, 3, 3, 1, 1, 1, compute)
        rows.append({"layer": name, "count_in_resnet56": count, "us": us, "us_with_pack": us_p, "us_cudnn_tf32": us_c,
                     "kernel": {3: "conv_tma_kernel<9>", 2: "conv_umma_kernel<9>"}.get(kind, str(kind)),
                     "TFLOPs": flop / us / 1e6, "io_GBs": byts / us / 1e3, "frac_hbm": byts / us / 1e3 / pk["hbm_gbs"]})
        tot_us += us * count; tot_cudnn += us_c * count; tot_flop += flop * count; tot_bytes += byts * count
    del flush
    torch.cuda.empty_cache()
    tma = compute == 2
    return {"bound": "hbm",
            "kernel": "po2::conv_tma_kernel<9> (tensor-map TMA producer, tcgen05 tf32)" if tma else "po2::conv_umma_kernel<9>",
            "unit": "GB/s",
            "achieved": tot_bytes / tot_us / 1e3, "peak": pk["hbm_gbs"], "frac": tot_bytes / tot_us / 1e3 / pk["hbm_gbs"],
            "traffic": 8.427e6 if tma else 8.43e6,
            "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of the 16->16 @32x32 layer under `ncu --set full` "
            "(profiles/r02_ncu_conv_tma_resnet56_16to16_3x3_at32_b128.csv): 8.427 MB read = the fp32 input exactly once (the "
            "halo rows of neighbouring tiles come out of L2), 0 B written back during the kernel (the 8.39 MB output is still "
            "dirty in the 126 MB L2 when the kernel ends); algorithmic bytes of that layer = 16.78 MB",
            "peak_source": pk["source"],
            "TFLOPs": tot_flop / tot_us / 1e6, "frac_of_bf16_peak": tot_flop / tot_us / 1e6 / pk["bf16_tflops"],
            "resnet56_3x3_forward_us": tot_us, "resnet56_3x3_forward_us_cudnn_tf32": tot_cudnn,
            "images_per_s_forward_qconv_only": batch / (tot_us * 1e-6), "layers": rows,
            "conv_operands": operand_label(ops.get_conv_mode()),
            "note": "the kernel family with the most launches and the largest share of the timed step (forward + data "
                    "gradient: 104 of 327 launches, profiles/r02_launches_*.csv); 52 stride-1 3x3 quantized convs of "
                    "ResNet-56 at batch %d, cold L2 (a 320 MB buffer is rewritten before every launch), CUDA-graph timed, the "
                    "launch the step performs (weight operand pre-packed by the step's multi-tensor quantizer launch); "
                    "algorithmic bytes per launch = 4*(B*C*H*W + B*K*P*Q).  These layers move 4-17 MB per launch: at the "
                    "measured HBM peak that is 0.6-2.6 us, of the order of a kernel launch itself" % batch}


# ------------------------------------------------------------------------------------------------
# the reference's CPU path
# ------------------------------------------------------------------------------------------------
def cpu_training_step_fn(batch):
    """The reference's training step on host cores: the one place bench.py executes the oracle / the
    staged reference files (as the baseline being timed, never as the product)."""
    torch.set_num_threads(os.cpu_count() or 1)
    return _reference_training_step(torch.device("cpu"), batch)


def cpu_baseline(batch, steps=2):
    step, loss_buf, kind, what, _ = cpu_training_step_fn(batch)
    step(); step()                          # first step: oneDNN primitive creation, thread-pool start-up
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return {"value": batch * steps / dt, "unit": "images/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"{steps} full training steps (fwd+bwd+SGD) of ResNet-56 PO2 4-bit QAT at batch {batch} after 2 warm-up "
                      f"steps; {what}",
            "ms_per_step": dt / steps * 1e3, "host_cpus": os.cpu_count()}


def run_reference(a):
    """--impl reference: the reference's own CPU implementation of the step on all host threads -- the
    unmodified reference files when baseline/_ref is staged, else the oracle's op-for-op torch port
    (pinned bit-exactly to the reference by tests/test_oracle_golden.py).  Same batch, same warm-up
    count, same number of timed steps and same config keys as our arm."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    B = a.batch
    step, loss_buf, kind, what, model = cpu_training_step_fn(B)
    warm = max(a.warmup, 3)
    for _ in range(warm):                    # the first one initialises the libraries
        step()
    steps = a.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    v = B * steps / dt
    sample = f"{steps} training steps at the full batch {B} after {warm} warm-up steps; {what}"
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": world,
           "steps": steps, "warmup": warm, "ms_per_step": dt / steps * 1e3, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32 (torch CPU kernels)",
           "data": DATA,
           "config": full_config(workload=WORKLOAD, batch_per_gpu=B, global_batch=B, device="cpu",
                                 parallelism="one process, %d host threads" % torch.get_num_threads(), cuda_graph=False,
                                 l2="n/a (CPU)", conv_backend="torch CPU (oneDNN) convolution", conv_operands="f32",
                                 norm_backend="torch CPU batch norm", weight_quantization="one quantizer call per layer (11 ATen ops each)",
                                 model_source=what, top1_identity="n/a (this arm is the reference)", bn_exchange_timeouts=0,
                                 last_loss=float(loss_buf.item())),
           "cpu_baseline": {"value": v, "unit": "images/s", "cores": torch.get_num_threads(), "kind": kind, "sample": sample},
           "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)
    if a.dump_outputs:
        dump_outputs(step_outputs(model, loss_buf), a.dump_outputs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=("ours", "reference"))
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sweep-log2", type=int, default=30, help="size of the quantizer roofline measurement")
    ap.add_argument("--sweep-max-log2", type=int, default=32, help="largest size of the compressed quantizer sweep")
    ap.add_argument("--parts", default="roofline,variants,oracle,configs,sweep",
                    help="N=1 only: which of the untimed side measurements to run (comma separated)")
    ap.add_argument("--torch-profile", default=None, help="write a torch.profiler kernel table of eager steps and exit")
    ap.add_argument("--graph-timeline", default=None, help="write the device timeline of graph replays (torch.profiler) and exit")
    ap.add_argument("--profile-step", action="store_true", help="run one eager step inside cudaProfilerStart/Stop and exit")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write the loss of the last step and the model's parameters and running "
                         "statistics after it as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
