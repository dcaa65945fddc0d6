"""torch.library custom ops over the C ABI.

Torch's role here is plumbing: it owns device memory and the current stream.  Every op enqueues
hand-written sm_100a kernels from libpo2b200.so on ``torch.cuda.current_stream()`` and is CUDA
graph capturable.  CPU tensors are rejected -- there is no fallback path.
"""
import os
from typing import Optional, Tuple

import torch

from . import _lib

_DT = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16, torch.float16: _lib.F16}
_FLAVORS = {"ieee": _lib.FLAVOR_IEEE, "torch_cpu": _lib.FLAVOR_IEEE, "torch_cuda": _lib.FLAVOR_TORCH_CUDA}
_flavor = _FLAVORS[os.environ.get("PO2_LOG2_FLAVOR", "ieee")]


def set_log2_flavor(name: str) -> None:
    """Which float-log2 the rounding boundaries reproduce: "ieee" (correctly rounded == torch CPU,
    the default and what the oracle uses) or "torch_cuda" (torch's CUDA kernels)."""
    global _flavor
    if name not in _FLAVORS:
        raise ValueError(f"unknown log2 flavor {name!r}; choose from {sorted(_FLAVORS)}")
    if _FLAVORS[name] == _lib.FLAVOR_TORCH_CUDA and not _lib.load().po2_have_torch_cuda_table():
        raise _lib.Po2Error("the torch_cuda boundary table has not been scanned into this build")
    _flavor = _FLAVORS[name]


def get_log2_flavor() -> str:
    return "torch_cuda" if _flavor == _lib.FLAVOR_TORCH_CUDA else "ieee"


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise _lib.Po2Error(f"{what}: po2_quantization_b200 runs on CUDA (sm_100a) only -- got a "
                            f"{t.device.type} tensor and there is no CPU fallback")
    if t.dtype not in _DT:
        raise TypeError(f"{what}: unsupported dtype {t.dtype} (float32, bfloat16, float16)")


def _aligned16(t: torch.Tensor) -> torch.Tensor:
    """t, or a copy of it when its data does not start on a 16-byte boundary.  A contiguous view can start at any
    element (``buf[1:].view(...)``); the tensor-core conv kernels read activations with 128-bit loads or tensor maps
    and the library refuses such a pointer (PO2_E_ALIGN), so the ops accept every input nn.Conv2d accepts."""
    return t if t.data_ptr() % 16 == 0 else t.clone()


_workspaces = {}

# ---- library paths taken instead of our kernels are never silent ------------------------------------
_noted = set()


def note_library_path(key: str, message: str) -> None:
    """A call that leaves the sm_100a kernels for a stock torch/cuDNN path says so: a warning the first
    time each distinct reason occurs, or a Po2Error when PO2_STRICT=1 (what the GPU test-suite and the
    benchmarks run with, so that a silent library fallback cannot pass for the product path)."""
    if os.environ.get("PO2_STRICT", "0") == "1":
        raise _lib.Po2Error(f"PO2_STRICT=1: {message}")
    if key not in _noted:
        _noted.add(key)
        import warnings
        warnings.warn(f"po2_quantization_b200: {message}", RuntimeWarning, stacklevel=3)


def release_workspaces() -> None:
    """Drop the per-(device, stream) scratch buffers (they are re-created on demand).  Call after the
    streams that used them are idle, e.g. between benchmark configurations."""
    _workspaces.clear()
    _dw_workspaces.clear()
    _wgrad_tickets.clear()
    from . import batchnorm
    batchnorm._bn_workspaces.clear()

# number of kernels of libpo2b200.so launched through this module (bench.py's `gpu_launches`)
LAUNCHES = 0


# "tf32" (default): tcgen05 tensor cores with tf32 operands -- the arithmetic of the reference's own cuDNN
# default on a GPU (activations keep 10 mantissa bits, PO2 weights exact); the stride-1 dense layers run on
# the TMA-fed kernel (csrc/po2_conv_tma.cuh: fp32 NCHW tiles staged by tensor-map TMA, no conversion pass).
# "tc": the register-fed kernel with bf16 operands (activations rounded to 8 mantissa bits; opt-in).
# "fp32": CUDA-core fp32 FMA everywhere (the fp32-accumulate parity mode); "cudnn": leave the convolution
# to F.conv2d.
COMPUTE = {"tc": 0, "fp32": 1, "tf32": 2}
E_SIZE = -4                    # PO2_E_SIZE: a tensor of 2^31 or more elements
DEFAULT_CONV_MODE = os.environ.get("PO2_CONV", "tf32")      # the mode of a fresh process (tests restore it)
_conv_mode = DEFAULT_CONV_MODE


def set_conv_mode(mode: str) -> None:
    global _conv_mode
    if mode not in ("tc", "tf32", "fp32", "cudnn"):
        raise ValueError("conv mode must be 'tc', 'tf32', 'fp32' or 'cudnn'")
    _conv_mode = mode


def get_conv_mode() -> str:
    return _conv_mode


def conv_backend_name() -> str:
    """Which kernel QuantizedConv2d's convolution runs on (reported by bench.py)."""
    return {"tc": "po2::conv_umma_kernel (tcgen05 bf16 implicit GEMM) / po2 depthwise+direct fp32 for the rest",
            "tf32": "po2::conv_umma_kernel (tcgen05 tf32 implicit GEMM) / po2 depthwise+direct fp32 for the rest",
            "fp32": "po2 CUDA-core fp32 kernels (depthwise / direct)",
            "cudnn": "cudnn (torch F.conv2d on the po2-quantized weight)"}[_conv_mode]


def _workspace(device: torch.device) -> torch.Tensor:
    """Zero-initialised scratch, one per (device, stream); the kernels leave it zeroed."""
    stream = torch.cuda.current_stream(device)
    key = (device.index, stream.cuda_stream)
    ws = _workspaces.get(key)
    if ws is None:
        ws = torch.zeros(int(_lib.load().po2_workspace_bytes()), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _code_bytes(n: int, bits: int) -> int:
    return (n + 1) // 2 if bits <= 4 else n


# ------------------------------------------------------------------------------------------------
# raw launchers (no autograd, no dispatcher) -- also what bench.py times
# ------------------------------------------------------------------------------------------------
def absmax_out(x: torch.Tensor, scale: torch.Tensor) -> None:
    global LAUNCHES
    lib = _lib.load()
    LAUNCHES += 1
    _lib.check(lib.po2_absmax(x.data_ptr(), x.numel(), _DT[x.dtype], scale.data_ptr(),
                              _workspace(x.device).data_ptr(), _stream_ptr(x.device)), "po2_absmax")


def quantize_out(x, y, scale, bits, fsr, plus, codes=None, zero_count=None, sse=None, flavor=None):
    global LAUNCHES
    lib = _lib.load()
    LAUNCHES += 1
    _lib.check(lib.po2_quantize(
        x.data_ptr(), y.data_ptr(), codes.data_ptr() if codes is not None else None,
        zero_count.data_ptr() if zero_count is not None else None,
        sse.data_ptr() if sse is not None else None, scale.data_ptr(), x.numel(), _DT[x.dtype],
        bits, fsr, int(plus), _flavor if flavor is None else flavor, _stream_ptr(x.device)), "po2_quantize")


def quantize_fused_out(x, y, scale, bits, fsr, plus, codes=None, zero_count=None, sse=None, flavor=None):
    global LAUNCHES
    lib = _lib.load()
    aligned = (x.data_ptr() | y.data_ptr()) % 16 == 0
    LAUNCHES += lib.po2_quantize_fused_launches(x.numel(), _DT[x.dtype]) if aligned else 2
    _lib.check(lib.po2_quantize_fused(
        x.data_ptr(), y.data_ptr(), codes.data_ptr() if codes is not None else None,
        zero_count.data_ptr() if zero_count is not None else None,
        sse.data_ptr() if sse is not None else None, scale.data_ptr(), x.numel(), _DT[x.dtype],
        bits, fsr, int(plus), _flavor if flavor is None else flavor,
        _workspace(x.device).data_ptr(), _stream_ptr(x.device)), "po2_quantize_fused")


# ------------------------------------------------------------------------------------------------
# custom ops
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("po2::quantize", mutates_args=(), device_types="cuda")
def quantize(x: torch.Tensor, bits: int, fsr: int, plus: bool) -> torch.Tensor:
    """y = 2^clamp(round(log2|x/s|)) * sign(x) * s, s = max|x| -- utils/quantizers.py:21-32, 41-52."""
    _require_cuda(x, "po2::quantize")
    x = x.contiguous()
    y = torch.empty_like(x)
    if x.numel() == 0:
        raise RuntimeError("max(): Expected reduction dim to be specified for input.numel() == 0")
    with torch.cuda.device(x.device):
        scale = torch.empty((), dtype=torch.float32, device=x.device)
        quantize_fused_out(x, y, scale, bits, fsr, plus)
    return y


@quantize.register_fake
def _(x, bits, fsr, plus):
    return torch.empty_like(x, memory_format=torch.contiguous_format)


def _quantize_bwd(ctx, grad):
    # straight-through estimator: utils/quantizers.py:34-36 returns grad_output itself
    return grad, None, None, None


quantize.register_autograd(_quantize_bwd)


@torch.library.custom_op("po2::quantize_full", mutates_args=(), device_types="cuda")
def quantize_full(x: torch.Tensor, bits: int, fsr: int, plus: bool
                  ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """(y, packed codes, scale, zero_count, sse): everything one pass over x can produce."""
    _require_cuda(x, "po2::quantize_full")
    x = x.contiguous()
    if x.numel() == 0:
        raise RuntimeError("max(): Expected reduction dim to be specified for input.numel() == 0")
    with torch.cuda.device(x.device):
        y = torch.empty_like(x)
        codes = torch.empty(_code_bytes(x.numel(), bits), dtype=torch.uint8, device=x.device)
        scale = torch.empty((), dtype=torch.float32, device=x.device)
        zero_count = torch.zeros((), dtype=torch.int32, device=x.device)
        sse = torch.zeros((), dtype=torch.float64, device=x.device)
        quantize_fused_out(x, y, scale, bits, fsr, plus, codes, zero_count, sse)
    return y, codes, scale, zero_count, sse


@quantize_full.register_fake
def _(x, bits, fsr, plus):
    n = x.numel()
    return (torch.empty_like(x, memory_format=torch.contiguous_format),
            x.new_empty(_code_bytes(n, bits), dtype=torch.uint8), x.new_empty((), dtype=torch.float32),
            x.new_empty((), dtype=torch.int32), x.new_empty((), dtype=torch.float64))


@torch.library.custom_op("po2::dequantize", mutates_args=(), device_types="cuda")
def dequantize(codes: torch.Tensor, scale: torch.Tensor, numel: int, bits: int, fsr: int,
               dtype: torch.dtype) -> torch.Tensor:
    """+-2^q * scale from packed sign+exponent codes."""
    if not codes.is_cuda:
        raise _lib.Po2Error("po2::dequantize: CUDA only")
    if dtype not in _DT:
        raise TypeError(f"po2::dequantize: unsupported dtype {dtype}")
    y = torch.empty(numel, dtype=dtype, device=codes.device)
    with torch.cuda.device(codes.device):
        _lib.check(_lib.load().po2_dequantize(codes.data_ptr(), scale.data_ptr(), y.data_ptr(), numel,
                                              _DT[dtype], bits, fsr, _stream_ptr(codes.device)),
                   "po2_dequantize")
    return y


@dequantize.register_fake
def _(codes, scale, numel, bits, fsr, dtype):
    return codes.new_empty(numel, dtype=dtype)


@torch.library.custom_op("po2::ste_backward", mutates_args=("grad_input",), device_types="cuda")
def ste_backward(grad_output: torch.Tensor, grad_input: torch.Tensor, accumulate: bool) -> None:
    """grad_input = grad_output (or += when accumulate) -- utils/quantizers.py:34-36, 54-56."""
    _require_cuda(grad_output, "po2::ste_backward")
    if grad_input.dtype != grad_output.dtype or grad_input.numel() != grad_output.numel():
        raise ValueError("po2::ste_backward: grad_input must match grad_output")
    if not (grad_output.is_contiguous() and grad_input.is_contiguous()):
        raise ValueError("po2::ste_backward: contiguous tensors only")
    with torch.cuda.device(grad_output.device):
        _lib.check(_lib.load().po2_ste_backward(grad_output.data_ptr(), grad_input.data_ptr(),
                                                grad_output.numel(), _DT[grad_output.dtype],
                                                int(accumulate), _stream_ptr(grad_output.device)),
                   "po2_ste_backward")


# ------------------------------------------------------------------------------------------------
# quantized-conv forward (models/quantized_conv.py:36,38)
# ------------------------------------------------------------------------------------------------
def conv2d_out(x, w, scale, out, stride, pad, groups, compute, w_format=_lib.W_F32_PO2, bits=4, fsr=1,
               wshape=None):
    """Raw launcher: out = conv2d(x, w).  w: fp32 (K, C/groups, R, S) on the grid +-scale*2^q, or the
    packed codes of such a tensor (w_format=W_CODES, wshape=(K, C/groups, R, S)).  x / out: fp32, or bf16 (inference
    of a bf16 model; w is then the exact fp32 widening of its bf16 weight)."""
    global LAUNCHES
    lib = _lib.load()
    check_conv_shapes(x.shape, w.shape if wshape is None else wshape, groups, pad)
    B, C, H, W_ = x.shape
    K, _, R, S = w.shape if wshape is None else wshape
    if w_format == _lib.W_CODES and w.numel() < _code_bytes(K * (C // groups) * R * S, bits):
        raise RuntimeError(f"po2 conv2d: {w.numel()} code bytes for a weight of shape {list(wshape)} at {bits} bits")
    dt = _DT[x.dtype]
    need = lib.po2_conv2d_workspace_dt(B, C, H, W_, K, R, S, stride, pad, groups, compute, dt)
    ws = torch.empty(max(int(need), 16), dtype=torch.uint8, device=x.device)
    fp32_w_bytes = (K * (C // groups) * R * S * 4 + 255) // 256 * 256
    LAUNCHES += (2 if need > fp32_w_bytes else 1) + (1 if w_format == _lib.W_CODES and need <= fp32_w_bytes else 0)
    _lib.check(lib.po2_conv2d_fwd_ep_dt(x.data_ptr(), w.data_ptr(), scale.data_ptr() if scale is not None else None,
                                        out.data_ptr(), B, C, H, W_, K, R, S, stride, pad, groups, w_format,
                                        bits, fsr, compute, ws.data_ptr(), ws.numel(), None, None, None, 0, dt,
                                        _stream_ptr(x.device)),
               "po2_conv2d_fwd")


def check_conv_shapes(xshape, wshape, groups: int, pad: int) -> None:
    """The argument errors nn.Conv2d / the reference raise (a RuntimeError, same wording as ATen) --
    the C ABI has no weight-channel argument, so a mismatch must be caught before the launch: the
    kernels would index K*(C/groups)*R*S weights past the end of a smaller buffer."""
    if len(xshape) != 4 or len(wshape) != 4:
        raise RuntimeError(f"Expected 4D (batched) input and 4D weight to conv2d, but got input of size: {list(xshape)} "
                           f"and weight of size: {list(wshape)}")
    B, C, H, W_ = xshape
    K, Cw, R, S = wshape
    if groups < 1 or K % groups != 0:
        raise RuntimeError(f"Given groups={groups}, expected weight to be divisible by {groups} at dimension 0, "
                           f"but got weight of size {list(wshape)}")
    if C != Cw * groups:
        raise RuntimeError(f"Given groups={groups}, weight of size {list(wshape)}, expected input{list(xshape)} to have "
                           f"{Cw * groups} channels, but got {C} channels instead")
    if H + 2 * pad < R or W_ + 2 * pad < S:
        raise RuntimeError(f"Calculated padded input size per channel: ({H + 2 * pad} x {W_ + 2 * pad}). Kernel size: "
                           f"({R} x {S}). Kernel size can't be greater than actual input size")


def conv_kernel_kind(xshape, wshape, stride: int, pad: int, groups: int, compute: int,
                     dtype: torch.dtype = torch.float32) -> int:
    """Which kernel conv2d runs for an input of shape xshape and dtype `dtype` (po2_conv2d_kernel_kind_dt, a planning
    query without a launch); negative: the PO2_E_* code the launch would return -- PO2_E_UNSUPPORTED for a bf16 shape
    that no bf16 kernel takes."""
    B, C, H, W_ = xshape
    K, _, R, S = wshape
    return int(_lib.load().po2_conv2d_kernel_kind_dt(B, C, H, W_, K, R, S, stride, pad, groups, compute, _DT[dtype]))


def _conv_weight(x, w, what):
    """w as the conv kernels take it: fp32 activations need fp32 weights; bf16 activations (a bf16 model at inference)
    take bf16 or fp32 weights, handed to the library as their exact fp32 widening"""
    if x.dtype == torch.float32 and w.dtype == torch.float32:
        return w
    if x.dtype == torch.bfloat16 and w.dtype in (torch.bfloat16, torch.float32):
        return w.float()
    raise TypeError(f"{what}: fp32 NCHW activations with fp32 weights, or bf16 NCHW activations (inference) only")


def _conv_out_shape(x, w, stride, pad):
    B, _, H, W_ = x.shape
    K, _, R, S = w.shape
    return (B, K, (H + 2 * pad - R) // stride + 1, (W_ + 2 * pad - S) // stride + 1)


@torch.library.custom_op("po2::conv2d", mutates_args=(), device_types="cuda")
def conv2d(x: torch.Tensor, w: torch.Tensor, scale: Optional[torch.Tensor], stride: int, pad: int,
           groups: int, compute: int) -> torch.Tensor:
    """conv2d(x, w) with w on the PO2 grid +-scale*2^q (scale=None: plain fp32 weights).
    compute 0: tcgen05 bf16 tensor cores (weights exact, activations rounded to bf16, fp32 accumulate)
    where the shape allows; 1: fp32 FMA everywhere.  A bf16 x (inference only) gives a bf16 output."""
    _require_cuda(x, "po2::conv2d")
    w = _conv_weight(x, w, "po2::conv2d")
    check_conv_shapes(x.shape, w.shape, groups, pad)
    x = _aligned16(x.contiguous())
    w = _aligned16(w.contiguous())
    out = torch.empty(_conv_out_shape(x, w, stride, pad), dtype=x.dtype, device=x.device)
    with torch.cuda.device(x.device):
        conv2d_out(x, w, scale, out, stride, pad, groups, compute)
    return out


@conv2d.register_fake
def _(x, w, scale, stride, pad, groups, compute):
    return x.new_empty(_conv_out_shape(x, w, stride, pad))


# "tc": data gradient of stride-1 dense convs on the tensor-core kernel (grad rounded to bf16, weights
# exact); "aten": everything through aten.convolution_backward (cuDNN)
_dgrad_mode = os.environ.get("PO2_CONV_DGRAD", "tc")


def set_dgrad_mode(mode: str) -> None:
    global _dgrad_mode
    if mode not in ("tc", "aten"):
        raise ValueError("dgrad mode must be 'tc' or 'aten'")
    _dgrad_mode = mode


def conv2d_dgrad_out(g, w, scale, gx, pad, compute: int = 0) -> bool:
    """gx = dL/dx of conv2d(x, w) (stride 1, dense) from g = dL/dout.  False if the shape is not taken."""
    global LAUNCHES
    lib = _lib.load()
    check_conv_shapes(gx.shape, w.shape, 1, pad)
    B, C, H, W_ = gx.shape
    K, _, R, S = w.shape
    if tuple(g.shape) != (B, K, H + 2 * pad - R + 1, W_ + 2 * pad - S + 1):
        raise RuntimeError(f"po2 conv2d dgrad: grad_output {list(g.shape)} does not match input {list(gx.shape)} / weight {list(w.shape)}")
    need = lib.po2_conv2d_dgrad_workspace(B, C, H, W_, K, R, S, pad, compute)
    if need == 0:
        return False
    ws = torch.empty(int(need), dtype=torch.uint8, device=g.device)
    rc = lib.po2_conv2d_dgrad(g.data_ptr(), w.data_ptr(), scale.data_ptr() if scale is not None else None,
                              gx.data_ptr(), B, C, H, W_, K, R, S, 1, pad, 1, _lib.W_F32_PO2, 4, 1, compute,
                              ws.data_ptr(), ws.numel(), _stream_ptr(g.device))
    if rc == -10:                      # PO2_E_UNSUPPORTED
        return False
    _lib.check(rc, "po2_conv2d_dgrad")
    LAUNCHES += 2
    return True


# "tc": weight gradient of stride-1 dense convs (K <= 128) on the tensor-core kernel (x and grad rounded
# to bf16, fp32 accumulation, deterministic), and of small wider 1x1 layers (B*H*W <= 8192, B*H*W*C*K <= 2^26) on
# the exact-fp32 CUDA-core GEMM (deterministic); "aten": aten.convolution_backward (cuDNN)
_wgrad_mode = os.environ.get("PO2_CONV_WGRAD", "tc")


def set_wgrad_mode(mode: str) -> None:
    global _wgrad_mode
    if mode not in ("tc", "aten"):
        raise ValueError("wgrad mode must be 'tc' or 'aten'")
    _wgrad_mode = mode


def conv2d_wgrad_out(g, x, gw, pad, compute: int = 0) -> bool:
    """gw = dL/dW of conv2d(x, W) (stride 1, dense) from g = dL/dout.  False if the shape is not taken.
    The library picks the kernel (po2_conv2d_wgrad_kernel_kind): 2 = K5T (tf32 operands, compute 2), 1 = K5 (bf16
    operands), 3 = the fp32 CUDA-core GEMM of 1x1 layers wider than K5T / K5 take, with B*H*W <= 8192 and
    B*H*W*C*K <= 2^26.  Each is the main kernel + the fixed-order reduce kernel (two launches)."""
    global LAUNCHES
    lib = _lib.load()
    check_conv_shapes(x.shape, gw.shape, 1, pad)
    B, C, H, W_ = x.shape
    K, _, R, S = gw.shape
    if tuple(g.shape) != (B, K, H + 2 * pad - R + 1, W_ + 2 * pad - S + 1):
        raise RuntimeError(f"po2 conv2d wgrad: grad_output {list(g.shape)} does not match input {list(x.shape)} / weight {list(gw.shape)}")
    need = lib.po2_conv2d_wgrad_workspace(B, C, H, W_, K, R, S, 1, pad, 1, compute)
    if need == 0:
        return False
    ws = torch.empty(int(need), dtype=torch.uint8, device=g.device)
    # 8 zeroed bytes per (device, stream): the grid barrier of the TMA-fed kernel's fused partial-sum reduction
    key = (g.device.index, torch.cuda.current_stream(g.device).cuda_stream)
    tk = _wgrad_tickets.get(key)
    if tk is None:
        tk = _wgrad_tickets[key] = torch.zeros(64, dtype=torch.uint8, device=g.device)
    rc = lib.po2_conv2d_wgrad_z(g.data_ptr(), x.data_ptr(), gw.data_ptr(), B, C, H, W_, K, R, S, 1, pad, 1, compute,
                                ws.data_ptr(), ws.numel(), tk.data_ptr(), _stream_ptr(g.device))
    if rc == -10:                      # PO2_E_UNSUPPORTED
        return False
    _lib.check(rc, "po2_conv2d_wgrad")
    fused = lib.po2_conv2d_wgrad_kernel_kind(B, C, H, W_, K, R, S, 1, pad, 1, compute) == 2 and \
        os.environ.get("PO2_WGRAD_FUSED_REDUCE", "0") == "1"
    LAUNCHES += 1 if fused else 2
    return True


def conv2d_dgrad_packed_out(g, packed, scale, gx, wshape, pad, compute) -> None:
    """gx = dL/dx from the data-gradient operand the forward's multi-tensor quantizer already packed: one launch"""
    global LAUNCHES
    B, C, H, W_ = gx.shape
    K, _, R, S = wshape
    LAUNCHES += 1
    _lib.check(_lib.load().po2_conv2d_dgrad_packed(g.data_ptr(), packed.data_ptr(), scale.data_ptr(), gx.data_ptr(),
                                                   B, C, H, W_, K, R, S, pad, compute, _stream_ptr(g.device)),
               "po2_conv2d_dgrad_packed")


def dilate2_out(g, g_up) -> None:
    """g_up[2p][2q] = g[p][q], zero elsewhere (the output gradient of a stride-2 conv at the input resolution)"""
    global LAUNCHES
    B, K, P, Q = g.shape
    LAUNCHES += 1
    _lib.check(_lib.load().po2_dilate2(g.data_ptr(), g_up.data_ptr(), B * K, P, Q, _stream_ptr(g.device)), "po2_dilate2")


def dilate2_into_out(g, g_up) -> None:
    """dilate2_out for any H x W of g_up with g's P x Q == ((H - 1) // 2 + 1, (W - 1) // 2 + 1): odd H or W, odd Q"""
    global LAUNCHES
    B, K, P, Q = g.shape
    H, W_ = g_up.shape[2:]
    LAUNCHES += 1
    _lib.check(_lib.load().po2_dilate2_into(g.data_ptr(), g_up.data_ptr(), B * K, P, Q, H, W_, _stream_ptr(g.device)),
               "po2_dilate2_into")


_dw_workspaces = {}
_wgrad_tickets = {}

# ---- weight gradients on a second stream --------------------------------------------------------------------
# The weight gradient of a layer is a leaf of the backward pass: nothing before the optimizer reads it.  With the
# overlap on, K5T / K5 / the pointwise GEMM (+ their reduce kernel) are launched on a per-device side stream that
# forks from the backward stream where the layer's output gradient exists, and the backward stream goes on to the
# data gradient and the norm kernels of the layers below; one join is queued on the autograd engine for the end of
# the backward pass.  Inside a CUDA-graph capture the side stream is a parallel branch of the graph.
_wgrad_overlap = os.environ.get("PO2_WGRAD_STREAM", "0") == "1"
_side_streams = {}
_side_pending = {}
_side_task = -1
_wgrad_trace = None                # tests: list that receives the data_ptr of every deferred gradient


def set_wgrad_overlap(on: bool) -> None:
    """Run the weight-gradient kernels of prefetched QuantizedConv2d layers on a side stream (joined at the end of
    backward()).  Only for training loops in which nothing reads a conv weight's gradient before backward()
    returns: the gradient tensor is handed to autograd while its kernel may still be running, which is safe when
    autograd installs it as ``weight.grad`` by reference (``zero_grad(set_to_none=True)``, no tensor hooks, no
    DistributedDataParallel reducer hooks); a layer whose weight already has a ``.grad`` is not deferred."""
    global _wgrad_overlap
    _wgrad_overlap = bool(on)


def get_wgrad_overlap() -> bool:
    return _wgrad_overlap


def join_weight_gradients() -> None:
    """Make the current stream (and the stream backward ran on) wait for the side stream's weight gradients.
    Queued automatically for the end of every backward pass that deferred one."""
    for side, main in list(_side_pending.values()):
        cur = torch.cuda.current_stream(side.device)
        cur.wait_stream(side)
        if main != cur:
            main.wait_stream(side)
    _side_pending.clear()


def side_stream(dev) -> "torch.cuda.Stream":
    side = _side_streams.get(dev.index)
    if side is None:
        side = _side_streams[dev.index] = torch.cuda.Stream(dev)     # lowest priority: the main branch goes first
    return side


def _wgrad_on_side_stream(g, x, gw, pad, compute, ready=None) -> bool:
    """ready: event on the backward stream after which g exists (default: everything queued so far)"""
    global _side_task
    dev = x.device
    side = side_stream(dev)
    main = torch.cuda.current_stream(dev)
    if ready is not None:
        side.wait_event(ready)
    else:
        side.wait_stream(main)
    with torch.cuda.stream(side):          # workspace and tickets belong to the side stream
        ok = conv2d_wgrad_out(g, x, gw, pad, compute)
    if not ok:
        return False
    # g and x are released by autograd on the backward stream while the side stream may still read them
    g.record_stream(side)
    x.record_stream(side)
    _side_pending[dev.index] = (side, main)
    task = torch._C._current_graph_task_id()
    if task != _side_task or task < 0:
        _side_task = task
        torch.autograd.Variable._execution_engine.queue_callback(join_weight_gradients)
    if _wgrad_trace is not None:
        _wgrad_trace.append(gw.data_ptr())
    return True


def _depthwise_backward(g_full, x, w, need_x, need_w):
    """(gx, gw) of a depthwise 3x3 pad-1 conv from the output gradient at the input resolution"""
    global LAUNCHES
    lib = _lib.load()
    B, C, H, W_ = x.shape
    gx = gw = None
    if need_x:
        gx = torch.empty_like(x)
        LAUNCHES += 1
        _lib.check(lib.po2_conv2d_depthwise_dgrad(g_full.data_ptr(), w.data_ptr(), gx.data_ptr(), B, C, H, W_,
                                                  _stream_ptr(x.device)), "po2_conv2d_depthwise_dgrad")
    if need_w:
        key = (x.device.index, torch.cuda.current_stream(x.device).cuda_stream)
        ws = _dw_workspaces.get(key)
        need = int(lib.po2_conv2d_depthwise_wgrad_workspace(4096))
        if ws is None:
            ws = _dw_workspaces[key] = torch.zeros(need, dtype=torch.uint8, device=x.device)
        gw = torch.empty_like(w)
        LAUNCHES += 1
        _lib.check(lib.po2_conv2d_depthwise_wgrad(g_full.data_ptr(), x.data_ptr(), gw.data_ptr(), B, C, H, W_,
                                                  ws.data_ptr(), ws.numel(), _stream_ptr(x.device)),
                   "po2_conv2d_depthwise_wgrad")
    return gx, gw


def _stride1_taken(B, C, H, W_, K, R, pad, compute, need_x, need_w) -> bool:
    """whether a kernel takes either gradient of the stride-1 problem on the zero-inserted output gradient (B, K, H, W)
    of a dense stride-2 layer.  The planner refuses it, among other reasons, when that gradient has 2^31 or more
    elements, which po2_dilate2 would refuse too: the layer then leaves the kernels before anything is dilated."""
    lib = _lib.load()
    return bool((need_x and lib.po2_conv2d_dgrad_workspace(B, C, H, W_, K, R, R, pad, compute) > 0) or
                (need_w and lib.po2_conv2d_wgrad_kernel_kind(B, C, H, W_, K, R, R, 1, pad, 1, compute) != 0))


def _conv_backward(g, x, w, scale, stride, pad, groups, compute, need_x, need_w, packed_d=None, defer_w=False):
    """(gx, gw) of conv2d(x, w) on our kernels: dense layers on the tcgen05 kernels (data gradient: the forward
    kernel with transposed weights; weight gradient: K5T / K5, or the fp32 GEMM for small wide 1x1 layers) --
    stride-2 layers through the zero-inserted output gradient, which turns both into stride-1 problems -- and
    depthwise 3x3 layers on the CUDA-core kernels of csrc/po2_conv_bwd.cu.  Whatever is left goes through aten.convolution_backward, loudly."""
    g = _aligned16(g.contiguous())
    x = _aligned16(x.contiguous())
    gx = gw = None
    B, C, H, W_ = x.shape
    K, _, R, S = w.shape
    fp32 = g.dtype == torch.float32 and x.dtype == torch.float32 and w.dtype == torch.float32
    ours = compute != 1 and groups == 1 and fp32 and stride in (1, 2)
    depthwise = (fp32 and _dgrad_mode == "tc" and groups == C == K and R == 3 and S == 3 and pad == 1 and stride in (1, 2)
                 and C <= 4096)
    # 3x3 pad 1 / 1x1 pad 0 at stride 2 is the stride-1 problem on the zero-inserted output gradient, at any H x W
    s2_ok = stride == 2 and ((R == 3 and pad == 1) or (R == 1 and pad == 0)) and \
        tuple(g.shape[2:]) == ((H - 1) // 2 + 1, (W_ - 1) // 2 + 1)
    with torch.cuda.device(x.device):
        g_s1 = g
        if stride == 2 and (ours or depthwise) and s2_ok and (need_x or need_w) and \
                (depthwise or _stride1_taken(B, C, H, W_, K, R, pad, compute, need_x, need_w)):
            g_s1 = torch.empty(B, K, H, W_, dtype=torch.float32, device=g.device)
            if H % 2 == 0 and W_ % 2 == 0 and g.shape[3] % 2 == 0:
                dilate2_out(g, g_s1)
            else:
                dilate2_into_out(g, g_s1)
        elif stride == 2:
            ours = depthwise = False
        if depthwise:
            gx, gw = _depthwise_backward(g_s1, x, w.contiguous(), need_x, need_w)
        else:
            defer_w = defer_w and _wgrad_overlap and need_w and ours and _wgrad_mode == "tc" and \
                torch._C._current_graph_task_id() >= 0
            ready = None
            if defer_w:
                # the side stream forks HERE (output gradient complete), not behind this layer's data gradient
                ready = torch.cuda.Event()
                ready.record(torch.cuda.current_stream(x.device))
            if need_x and ours and _dgrad_mode == "tc" and scale is not None:
                cand = torch.empty_like(x)
                if packed_d is not None and stride == 1:
                    conv2d_dgrad_packed_out(g_s1, packed_d, scale, cand, w.shape, pad, compute)
                    gx = cand
                elif conv2d_dgrad_out(g_s1, w, scale, cand, pad, compute):
                    gx = cand
            if need_w and ours and _wgrad_mode == "tc":
                cand = torch.empty_like(w)
                # tf32 mode: the TMA-fed tf32 kernel where the shape allows; elsewhere the library takes the
                # bf16-operand kernel (the weight gradient is a leaf of the backward pass: its rounding does not
                # propagate into other layers' gradients, unlike the data gradient)
                if defer_w:
                    if _wgrad_on_side_stream(g_s1, x, cand, pad, compute, ready):
                        gw = cand
                elif conv2d_wgrad_out(g_s1, x, cand, pad, compute):
                    gw = cand
    if (need_x and gx is None) or (need_w and gw is None):
        if x.is_cuda and _conv_mode != "cudnn":
            note_library_path("conv_backward_aten",
                              f"convolution backward of input {list(x.shape)} / weight {list(w.shape)} stride {stride} groups "
                              f"{groups} runs on aten.convolution_backward (cuDNN): shape not taken by the po2 kernels")
        gx2, gw2, _ = torch.ops.aten.convolution_backward(
            g, x, w, None, [stride, stride], [pad, pad], [1, 1], False, [0, 0], groups,
            [need_x and gx is None, need_w and gw is None, False])
        gx = gx if gx is not None else gx2
        gw = gw if gw is not None else gw2
    return gx, gw


def _no_bf16_backward(x, what):
    if x.dtype == torch.bfloat16:
        raise RuntimeError(f"{what}: a bf16 convolution runs at inference only -- there is no bf16 backward; run it under "
                           "torch.no_grad() / torch.inference_mode(), or train in fp32")


def _conv2d_setup(ctx, inputs, output):
    x, w, scale, stride, pad, groups, compute = inputs
    _no_bf16_backward(x, "po2::conv2d")
    ctx.save_for_backward(x, w, scale) if scale is not None else ctx.save_for_backward(x, w)
    ctx.has_scale = scale is not None
    ctx.cfg = (stride, pad, groups, compute)


def _conv2d_bwd(ctx, g):
    saved = ctx.saved_tensors
    x, w = saved[0], saved[1]
    scale = saved[2] if ctx.has_scale else None
    stride, pad, groups, compute = ctx.cfg
    gx, gw = _conv_backward(g, x, w, scale, stride, pad, groups, compute, ctx.needs_input_grad[0],
                            ctx.needs_input_grad[1])
    return gx, gw, None, None, None, None, None


conv2d.register_autograd(_conv2d_bwd, setup_context=_conv2d_setup)


@torch.library.custom_op("po2::quantize_scaled", mutates_args=(), device_types="cuda")
def quantize_scaled(x: torch.Tensor, bits: int, fsr: int, plus: bool) -> Tuple[torch.Tensor, torch.Tensor]:
    """(y, scale): the quantized tensor and its per-tensor max-abs scale (what the conv needs to
    rebuild the exact +-2^q operand)."""
    _require_cuda(x, "po2::quantize_scaled")
    x = x.contiguous()
    if x.numel() == 0:
        raise RuntimeError("max(): Expected reduction dim to be specified for input.numel() == 0")
    with torch.cuda.device(x.device):
        y = torch.empty_like(x)
        scale = torch.empty((), dtype=torch.float32, device=x.device)
        quantize_fused_out(x, y, scale, bits, fsr, plus)
    return y, scale


@quantize_scaled.register_fake
def _(x, bits, fsr, plus):
    return torch.empty_like(x, memory_format=torch.contiguous_format), x.new_empty((), dtype=torch.float32)


def _quantize_scaled_bwd(ctx, gy, gscale):
    return gy, None, None, None          # straight-through (utils/quantizers.py:34-36)


quantize_scaled.register_autograd(_quantize_scaled_bwd)


# ------------------------------------------------------------------------------------------------
# QAT forward as one op: quantize the master weight + convolve (models/quantized_conv.py:34-36)
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("po2::qconv2d", mutates_args=(), device_types="cuda")
def qconv2d(x: torch.Tensor, weight: torch.Tensor, bits: int, fsr: int, plus: bool, stride: int, pad: int,
            groups: int, compute: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """(out, quantized weight, scale) = conv2d(x, Q(weight)).  The quantizer kernel emits the conv's
    packed bf16 operand directly where the shape allows, so the forward is two kernel launches."""
    global LAUNCHES
    _require_cuda(x, "po2::qconv2d")
    if x.dtype != torch.float32 or weight.dtype != torch.float32:
        raise TypeError("po2::qconv2d: fp32 NCHW activations and fp32 weights only")
    check_conv_shapes(x.shape, weight.shape, groups, pad)
    x = _aligned16(x.contiguous())
    w = weight.contiguous()
    lib = _lib.load()
    B, C, H, W_ = x.shape
    K, _, R, S = w.shape
    out = torch.empty(_conv_out_shape(x, w, stride, pad), dtype=torch.float32, device=x.device)
    qw = torch.empty_like(w)
    scale = torch.empty((), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        need = lib.po2_conv2d_workspace(B, C, H, W_, K, R, S, stride, pad, groups, compute)
        ws = torch.empty(max(int(need), 16), dtype=torch.uint8, device=x.device)
        LAUNCHES += 3 if (C % 16 or K % 16 or groups != 1) else 2
        _lib.check(lib.po2_qconv2d_fwd(x.data_ptr(), w.data_ptr(), qw.data_ptr(), scale.data_ptr(), out.data_ptr(),
                                       B, C, H, W_, K, R, S, stride, pad, groups, bits, fsr, int(plus), _flavor,
                                       compute, ws.data_ptr(), ws.numel(), _workspace(x.device).data_ptr(),
                                       _stream_ptr(x.device)), "po2_qconv2d_fwd")
    return out, qw, scale


@qconv2d.register_fake
def _(x, weight, bits, fsr, plus, stride, pad, groups, compute):
    return (x.new_empty(_conv_out_shape(x, weight, stride, pad)), torch.empty_like(weight, memory_format=torch.contiguous_format),
            x.new_empty((), dtype=torch.float32))


def _qconv2d_setup(ctx, inputs, output):
    x, weight, bits, fsr, plus, stride, pad, groups, compute = inputs
    out, qw, scale = output
    ctx.save_for_backward(x, qw, scale)
    ctx.cfg = (stride, pad, groups, compute)
    # qw / scale are normally unused downstream: do not let autograd manufacture zero gradients for
    # them (two fill kernels and an add per layer and step)
    ctx.set_materialize_grads(False)


def _qconv2d_bwd(ctx, g, g_qw, g_scale):
    x, qw, scale = ctx.saved_tensors
    stride, pad, groups, compute = ctx.cfg
    need_x, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
    if g is None:                            # only the quantized weight was used: straight-through
        return None, g_qw, None, None, None, None, None, None, None
    gx, gw = _conv_backward(g, x, qw, scale, stride, pad, groups, compute, need_x, need_w)
    if g_qw is not None and gw is not None:
        gw = gw + g_qw                       # someone also used the returned quantized weight
    elif g_qw is not None:
        gw = g_qw
    # straight-through estimator (utils/quantizers.py:34-36): d/d weight == d/d quantized weight
    return gx, gw, None, None, None, None, None, None, None


qconv2d.register_autograd(_qconv2d_bwd, setup_context=_qconv2d_setup)


# ------------------------------------------------------------------------------------------------
# lin / lin+ QAT forward (utils/quantizers.py:59-136 + models/quantized_conv.py:34-36).  A lin weight is n * 2^k per
# input channel (|n| <= 2^(bits-1) - 1), so it is its own exact tensor-core operand up to these bit widths; every
# consumer of (packed, scale) then takes it with scale = 1.0.
# ------------------------------------------------------------------------------------------------
LIN_EXACT_BITS = {"tc": 9, "tf32": 12, "fp32": 16}
LIN_ITERS = 10                     # utils/quantizers.py: num_iters default, what QuantizedConv2d and quantize_model use
_ones = {}


def lin_scale(device) -> torch.Tensor:
    """the per-device fp32 1.0 that stands for the scale of a lin operand (created on first use, outside a capture)"""
    one = _ones.get(device.index)
    if one is None:
        one = _ones[device.index] = torch.ones((), dtype=torch.float32, device=device)
    return one


@torch.library.custom_op("po2::lin_qconv2d", mutates_args=(), device_types="cuda")
def lin_qconv2d(x: torch.Tensor, weight: torch.Tensor, bits: int, plus: bool, stride: int, pad: int, groups: int,
                compute: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """(out, y) = (conv2d(x, y), y) with y = lin(weight) (lin+ with plus): the quantizer kernel also writes the conv's
    packed operand where the shape has one, so the forward is two launches; elsewhere (depthwise, small pointwise,
    compute 1) the CUDA-core kernels read y directly."""
    global LAUNCHES
    _require_cuda(x, "po2::lin_qconv2d")
    if x.dtype != torch.float32 or weight.dtype != torch.float32:
        raise TypeError("po2::lin_qconv2d: fp32 NCHW activations and fp32 weights only")
    check_conv_shapes(x.shape, weight.shape, groups, pad)
    x = _aligned16(x.contiguous())
    w = weight.contiguous()
    lib = _lib.load()
    B, C, H, W_ = x.shape
    K, Cg, R, S = w.shape
    out = torch.empty(_conv_out_shape(x, w, stride, pad), dtype=torch.float32, device=x.device)
    y = torch.empty_like(w)
    with torch.cuda.device(x.device):
        one = lin_scale(x.device)
        st = _stream_ptr(x.device)
        nbytes = int(lib.po2_conv2d_pack_bytes(B, C, H, W_, K, R, S, stride, pad, groups, compute))
        if nbytes:
            packed = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
            LAUNCHES += 2 if (C % 16 == 0 and K % 16 == 0) else 3
            _lib.check(lib.po2_lin_quantize_pack(w.data_ptr(), y.data_ptr(), packed.data_ptr(), nbytes, None, 0, B, C, H, W_,
                                                 K, R, S, stride, pad, groups, int(bits), LIN_ITERS, int(plus), _flavor,
                                                 compute, st), "po2_lin_quantize_pack")
            _lib.check(lib.po2_conv2d_fwd_packed(x.data_ptr(), packed.data_ptr(), one.data_ptr(), out.data_ptr(), B, C, H,
                                                 W_, K, R, S, stride, pad, groups, compute, st), "po2_conv2d_fwd_packed")
        else:
            LAUNCHES += 1
            _lib.check(lib.po2_lin_quantize(w.data_ptr(), y.data_ptr(), K, Cg, R * S, int(bits), LIN_ITERS, int(plus),
                                            _flavor, st), "po2_lin_quantize")
            conv2d_out(x, y, one, out, stride, pad, groups, compute)
    return out, y


@lin_qconv2d.register_fake
def _(x, weight, bits, plus, stride, pad, groups, compute):
    return x.new_empty(_conv_out_shape(x, weight, stride, pad)), torch.empty_like(weight, memory_format=torch.contiguous_format)


def _lin_qconv2d_setup(ctx, inputs, output):
    x, weight, bits, plus, stride, pad, groups, compute = inputs
    out, y = output
    ctx.save_for_backward(x, y)
    ctx.cfg = (stride, pad, groups, compute)
    ctx.set_materialize_grads(False)


def _lin_qconv2d_bwd(ctx, g, g_y):
    x, y = ctx.saved_tensors
    stride, pad, groups, compute = ctx.cfg
    if g is None:                            # only the quantized weight was used: straight-through
        return None, g_y, None, None, None, None, None, None
    gx, gw = _conv_backward(g, x, y, lin_scale(x.device), stride, pad, groups, compute, ctx.needs_input_grad[0],
                            ctx.needs_input_grad[1])
    if g_y is not None:
        gw = g_y if gw is None else gw + g_y
    # straight-through estimator (utils/quantizers.py:94-96): d/d weight == d/d quantized weight
    return gx, gw, None, None, None, None, None, None


lin_qconv2d.register_autograd(_lin_qconv2d_bwd, setup_context=_lin_qconv2d_setup)


# ------------------------------------------------------------------------------------------------
# static weights: pack once, then one launch per forward
# ------------------------------------------------------------------------------------------------
def conv2d_pack(w: torch.Tensor, scale: Optional[torch.Tensor], xshape, stride: int, pad: int, groups: int,
                compute: int = 0, xdtype: torch.dtype = torch.float32):
    """Packed bf16 tensor-core operand for conv2d(x of shape xshape and dtype xdtype, w), or None if that shape does not
    run on the tensor-core kernel.  w: fp32, or (bf16 x) the model's bf16 weight, packed from its exact fp32 widening."""
    global LAUNCHES
    lib = _lib.load()
    check_conv_shapes(xshape, w.shape, groups, pad)
    B, C, H, W_ = xshape
    K, _, R, S = w.shape
    dt = _DT[xdtype]
    nbytes = lib.po2_conv2d_pack_bytes_dt(B, C, H, W_, K, R, S, stride, pad, groups, compute, dt)
    if nbytes == 0:
        return None
    w = w.float().contiguous()
    packed = torch.empty(int(nbytes), dtype=torch.uint8, device=w.device)
    with torch.cuda.device(w.device):
        LAUNCHES += 1
        _lib.check(lib.po2_conv2d_pack_dt(w.data_ptr(), scale.data_ptr() if scale is not None else None, packed.data_ptr(),
                                          packed.numel(), B, C, H, W_, K, R, S, stride, pad, groups, _lib.W_F32_PO2, 4, 1,
                                          compute, dt, _stream_ptr(w.device)), "po2_conv2d_pack")
    return packed


@torch.library.custom_op("po2::conv2d_packed", mutates_args=(), device_types="cuda")
def conv2d_packed(x: torch.Tensor, packed: torch.Tensor, scale: Optional[torch.Tensor], K: int, R: int, S: int,
                  stride: int, pad: int, groups: int, compute: int) -> torch.Tensor:
    """conv2d from a pre-packed weight operand (inference with static weights): one kernel launch.  x: fp32, or bf16
    (the operand packed for a bf16 x); the output has x's dtype."""
    global LAUNCHES
    _require_cuda(x, "po2::conv2d_packed")
    if x.dim() != 4:
        raise RuntimeError(f"Expected 4D (batched) input to conv2d, but got input of size: {list(x.shape)}")
    x = _aligned16(x.contiguous())
    B, C, H, W_ = x.shape
    dt = _act_dt(x, "po2::conv2d_packed")
    # the packed operand was laid out for ONE (input shape, weight shape): re-validate it against this input
    need = int(_lib.load().po2_conv2d_pack_bytes_dt(B, C, H, W_, K, R, S, stride, pad, groups, compute, dt))
    if need == 0 or packed.numel() != need:
        raise RuntimeError(f"po2::conv2d_packed: the packed operand ({packed.numel()} bytes) was not built for input "
                           f"{list(x.shape)} / weight [{K}, {C // max(groups, 1)}, {R}, {S}] (needs {need} bytes)")
    out = torch.empty((B, K, (H + 2 * pad - R) // stride + 1, (W_ + 2 * pad - S) // stride + 1),
                      dtype=x.dtype, device=x.device)
    with torch.cuda.device(x.device):
        LAUNCHES += 1
        _lib.check(_lib.load().po2_conv2d_fwd_packed_ep_dt(x.data_ptr(), packed.data_ptr(),
                                                           scale.data_ptr() if scale is not None else None, out.data_ptr(),
                                                           B, C, H, W_, K, R, S, stride, pad, groups, compute,
                                                           None, None, None, 0, dt, _stream_ptr(x.device)),
                   "po2_conv2d_fwd_packed")
    return out


@conv2d_packed.register_fake
def _(x, packed, scale, K, R, S, stride, pad, groups, compute):
    B, C, H, W_ = x.shape
    return x.new_empty((B, K, (H + 2 * pad - R) // stride + 1, (W_ + 2 * pad - S) // stride + 1))


# ------------------------------------------------------------------------------------------------
# inference with eval-mode BatchNorm (+ residual add) (+ activation) folded into the conv's epilogue
# ------------------------------------------------------------------------------------------------
def _act_dt(x, what):
    """the C ABI dtype of a conv's activations: fp32, or bf16 (inference)"""
    if x.dtype not in (torch.float32, torch.bfloat16):
        raise TypeError(f"{what}: fp32 or bf16 NCHW activations only, got {x.dtype}")
    return _DT[x.dtype]


def _ep_check(out, K, ep_a, ep_b, residual):
    out_shape = out.shape
    if ep_a.numel() != K or ep_b.numel() != K or ep_a.dtype != torch.float32 or ep_b.dtype != torch.float32:
        raise RuntimeError(f"po2 conv epilogue: scale/shift must be fp32 vectors of {K} out channels")
    if residual is not None and (tuple(residual.shape) != tuple(out_shape) or residual.dtype != out.dtype):
        raise RuntimeError(f"po2 conv epilogue: residual {list(residual.shape)} does not match the output {list(out_shape)}")


@torch.library.custom_op("po2::conv2d_packed_ep", mutates_args=(), device_types="cuda")
def conv2d_packed_ep(x: torch.Tensor, packed: torch.Tensor, scale: Optional[torch.Tensor], K: int, R: int, S: int,
                     stride: int, pad: int, groups: int, compute: int, ep_a: torch.Tensor, ep_b: torch.Tensor,
                     residual: Optional[torch.Tensor], act: int) -> torch.Tensor:
    """act(conv2d(x, W) * ep_a[k] + ep_b[k] + residual) from a pre-packed weight operand: one launch (inference)."""
    global LAUNCHES
    _require_cuda(x, "po2::conv2d_packed_ep")
    x = _aligned16(x.contiguous())
    B, C, H, W_ = x.shape
    dt = _act_dt(x, "po2::conv2d_packed_ep")
    need = int(_lib.load().po2_conv2d_pack_bytes_dt(B, C, H, W_, K, R, S, stride, pad, groups, compute, dt))
    if need == 0 or packed.numel() != need:
        raise RuntimeError(f"po2::conv2d_packed_ep: the packed operand ({packed.numel()} bytes) was not built for input "
                           f"{list(x.shape)} / weight [{K}, {C // max(groups, 1)}, {R}, {S}] (needs {need} bytes)")
    out = torch.empty((B, K, (H + 2 * pad - R) // stride + 1, (W_ + 2 * pad - S) // stride + 1),
                      dtype=x.dtype, device=x.device)
    _ep_check(out, K, ep_a, ep_b, residual)
    if residual is not None:
        residual = residual.contiguous()
    with torch.cuda.device(x.device):
        LAUNCHES += 1
        _lib.check(_lib.load().po2_conv2d_fwd_packed_ep_dt(
            x.data_ptr(), packed.data_ptr(), scale.data_ptr() if scale is not None else None, out.data_ptr(),
            B, C, H, W_, K, R, S, stride, pad, groups, compute, ep_a.data_ptr(), ep_b.data_ptr(),
            residual.data_ptr() if residual is not None else None, int(act), dt, _stream_ptr(x.device)),
            "po2_conv2d_fwd_packed_ep")
    return out


@conv2d_packed_ep.register_fake
def _(x, packed, scale, K, R, S, stride, pad, groups, compute, ep_a, ep_b, residual, act):
    B, C, H, W_ = x.shape
    return x.new_empty((B, K, (H + 2 * pad - R) // stride + 1, (W_ + 2 * pad - S) // stride + 1))


@torch.library.custom_op("po2::conv2d_ep", mutates_args=(), device_types="cuda")
def conv2d_ep(x: torch.Tensor, w: torch.Tensor, scale: Optional[torch.Tensor], stride: int, pad: int, groups: int,
              compute: int, ep_a: torch.Tensor, ep_b: torch.Tensor, residual: Optional[torch.Tensor],
              act: int) -> torch.Tensor:
    """act(conv2d(x, w) * ep_a[k] + ep_b[k] + residual) for any layer kind (depthwise, direct, tensor-core with an
    inline pack): inference only.  A bf16 x (with a bf16 residual) gives a bf16 output."""
    global LAUNCHES
    _require_cuda(x, "po2::conv2d_ep")
    w = _conv_weight(x, w, "po2::conv2d_ep")
    check_conv_shapes(x.shape, w.shape, groups, pad)
    x = _aligned16(x.contiguous())
    w = _aligned16(w.contiguous())
    lib = _lib.load()
    B, C, H, W_ = x.shape
    K, _, R, S = w.shape
    dt = _DT[x.dtype]
    out = torch.empty(_conv_out_shape(x, w, stride, pad), dtype=x.dtype, device=x.device)
    _ep_check(out, K, ep_a, ep_b, residual)
    if residual is not None:
        residual = residual.contiguous()
    with torch.cuda.device(x.device):
        need = lib.po2_conv2d_workspace_dt(B, C, H, W_, K, R, S, stride, pad, groups, compute, dt)
        ws = torch.empty(max(int(need), 16), dtype=torch.uint8, device=x.device)
        fp32_w_bytes = (K * (C // groups) * R * S * 4 + 255) // 256 * 256
        LAUNCHES += 2 if need > fp32_w_bytes else 1
        _lib.check(lib.po2_conv2d_fwd_ep_dt(x.data_ptr(), w.data_ptr(), scale.data_ptr() if scale is not None else None,
                                            out.data_ptr(), B, C, H, W_, K, R, S, stride, pad, groups, _lib.W_F32_PO2, 4,
                                            1, compute, ws.data_ptr(), ws.numel(), ep_a.data_ptr(), ep_b.data_ptr(),
                                            residual.data_ptr() if residual is not None else None, int(act), dt,
                                            _stream_ptr(x.device)), "po2_conv2d_fwd_ep")
    return out


@conv2d_ep.register_fake
def _(x, w, scale, stride, pad, groups, compute, ep_a, ep_b, residual, act):
    return x.new_empty(_conv_out_shape(x, w, stride, pad))
