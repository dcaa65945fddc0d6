"""ctypes binding of libpo2b200.so (the C ABI declared in include/po2_b200.h).

There is no fallback: if the library is missing and cannot be built, or a call fails, this
raises.  torch is used by callers only for device memory and streams.
"""
import ctypes
import os
import threading

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libpo2b200.so")

F32, BF16, F16 = 0, 1, 2
MODE_PO2, MODE_PO2_PLUS = 0, 1
FLAVOR_IEEE, FLAVOR_TORCH_CUDA = 0, 1
W_F32_PO2, W_CODES = 0, 1

_c = ctypes
_vp, _i, _i64, _sz = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_size_t

# name -> (restype, argtypes); must list every symbol include/po2_b200.h declares
SIGNATURES = {
    "po2_abi_version": (_i, []),
    "po2_error_string": (_c.c_char_p, [_i]),
    "po2_have_torch_cuda_table": (_i, []),
    "po2_workspace_bytes": (_sz, []),
    "po2_absmax": (_i, [_vp, _i64, _i, _vp, _vp, _vp]),
    "po2_quantize": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _i, _i, _i, _vp]),
    "po2_quantize_fused": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _i, _i, _i, _vp, _vp]),
    "po2_quantize_fused_launches": (_i, [_i64, _i]),
    "po2_dequantize": (_i, [_vp, _vp, _vp, _i64, _i, _i, _i, _vp]),
    "po2_ste_backward": (_i, [_vp, _vp, _i64, _i, _i, _vp]),
    "po2_conv2d_workspace": (_sz, [_i] * 11),
    "po2_conv2d_kernel_kind": (_i, [_i] * 11),
    "po2_conv2d_fwd": (_i, [_vp, _vp, _vp, _vp] + [_i] * 14 + [_vp, _sz, _vp]),
    "po2_conv2d_fwd_ep": (_i, [_vp, _vp, _vp, _vp] + [_i] * 14 + [_vp, _sz, _vp, _vp, _vp, _i, _vp]),
    "po2_conv2d_fwd_packed_ep": (_i, [_vp] * 4 + [_i] * 11 + [_vp, _vp, _vp, _i, _vp]),
    "po2_conv2d_pack_bytes": (_sz, [_i] * 11),
    "po2_conv2d_pack": (_i, [_vp, _vp, _vp, _sz] + [_i] * 14 + [_vp]),
    "po2_conv2d_fwd_packed": (_i, [_vp] * 4 + [_i] * 11 + [_vp]),
    "po2_conv2d_workspace_dt": (_sz, [_i] * 12),
    "po2_conv2d_kernel_kind_dt": (_i, [_i] * 12),
    "po2_conv2d_pack_bytes_dt": (_sz, [_i] * 12),
    "po2_conv2d_pack_dt": (_i, [_vp, _vp, _vp, _sz] + [_i] * 15 + [_vp]),
    "po2_conv2d_fwd_ep_dt": (_i, [_vp, _vp, _vp, _vp] + [_i] * 14 + [_vp, _sz, _vp, _vp, _vp, _i, _i, _vp]),
    "po2_conv2d_fwd_packed_ep_dt": (_i, [_vp] * 4 + [_i] * 11 + [_vp, _vp, _vp, _i, _i, _vp]),
    "po2_qconv2d_fwd": (_i, [_vp] * 5 + [_i] * 15 + [_vp, _sz, _vp, _vp]),
    "po2_quantize_pack": (_i, [_vp, _vp, _vp, _vp, _sz] + [_i] * 15 + [_vp, _vp]),
    "po2_multi_desc_bytes": (_sz, []),
    "po2_multi_desc_fill": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _sz] + [_i] * 15 + [_vp]),
    "po2_quantize_pack_multi": (_i, [_vp, _i, _i, _vp]),
    "po2_conv2d_dgrad_pack_bytes": (_sz, [_i] * 9),
    "po2_multi_desc_fill_dgrad": (_i, [_vp, _i, _vp, _sz] + [_i] * 11),
    "po2_conv2d_dgrad_packed": (_i, [_vp] * 4 + [_i] * 9 + [_vp]),
    "po2_conv2d_dgrad_workspace": (_sz, [_i] * 9),
    "po2_conv2d_dgrad": (_i, [_vp, _vp, _vp, _vp] + [_i] * 14 + [_vp, _sz, _vp]),
    "po2_dilate2": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "po2_dilate2_into": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "po2_conv2d_stem_wgrad_workspace": (_sz, [_i] * 10),
    "po2_conv2d_stem_wgrad": (_i, [_vp, _vp, _vp] + [_i] * 10 + [_vp, _sz, _vp]),
    "po2_sgd_step": (_i, [_vp, _vp, _vp, _vp, _i, _c.c_float, _c.c_float, _c.c_float, _i, _vp]),
    "po2_sgd_max_tensors_per_launch": (_i, []),
    "po2_conv2d_depthwise_dgrad": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "po2_conv2d_depthwise_wgrad_workspace": (_sz, [_i]),
    "po2_conv2d_depthwise_wgrad": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _sz, _vp]),
    "po2_conv2d_wgrad_workspace": (_sz, [_i] * 11),
    "po2_conv2d_wgrad_kernel_kind": (_i, [_i] * 11),
    "po2_conv2d_wgrad_z": (_i, [_vp, _vp, _vp] + [_i] * 11 + [_vp, _sz, _vp, _vp]),
    "po2_conv2d_wgrad": (_i, [_vp, _vp, _vp] + [_i] * 11 + [_vp, _sz, _vp]),
    "po2_lin_max_channel_elems": (_i, []),
    "po2_lin_quantize": (_i, [_vp, _vp] + [_i] * 7 + [_vp]),
    "po2_lin_quantize_dt": (_i, [_vp, _vp] + [_i] * 8 + [_vp]),
    "po2_lin_quantize_pack": (_i, [_vp, _vp, _vp, _sz, _vp, _sz] + [_i] * 15 + [_vp]),
    "po2_lin_multi_desc_bytes": (_sz, []),
    "po2_lin_multi_desc_fill": (_i, [_vp, _i, _vp, _vp, _vp, _sz, _vp, _sz] + [_i] * 15),
    "po2_lin_quantize_pack_multi": (_i, [_vp, _i, _i, _i, _vp]),
    "po2_bn_workspace_bytes": (_sz, [_i]),
    "po2_bn_mailbox_bytes": (_sz, []),
    "po2_bn_stats": (_i, [_vp, _i, _i, _i, _vp, _vp, _sz, _vp, _i, _i, _vp]),
    "po2_bn_apply": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _c.c_float, _c.c_float,
                          _i, _i, _vp, _vp, _i, _i, _i, _vp]),
    "po2_bn_fwd_fused": (_i, [_vp] * 8 + [_c.c_float, _c.c_float, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _sz, _vp, _i, _i, _vp]),
    "po2_bn_bwd_fused": (_i, [_vp] * 12 + [_i] * 4 + [_vp, _sz, _vp]),
    "po2_bn_bwd_reduce": (_i, [_vp] * 11 + [_i] * 4 + [_vp, _sz, _vp, _i, _i, _vp]),
    "po2_bn_bwd_apply": (_i, [_vp] * 10 + [_i, _vp, _vp, _vp] + [_i] * 4 + [_vp]),
}

_lock = threading.Lock()
_lib = None


class Po2Error(RuntimeError):
    pass


def load():
    """Load (building first if the .so is absent) and type the library.  Raises on failure."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            from . import build as _build
            _build.build()
        try:
            lib = ctypes.CDLL(LIB_PATH)
        except OSError as e:  # pragma: no cover
            raise Po2Error(f"cannot load {LIB_PATH}: {e}. Run `python -m po2_quantization_b200.build`; "
                           "there is no CPU or PyTorch fallback for this path.") from e
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)     # AttributeError if the ABI and the header disagree
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(code: int, what: str):
    if code != 0:
        msg = load().po2_error_string(code).decode()
        raise Po2Error(f"{what} failed ({code}): {msg}")
