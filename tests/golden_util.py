"""Helpers to read the committed golden fixtures (bit patterns -> values)."""
import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    return np.load(os.path.join(GOLDEN_DIR, name))


def bits_to_f32(u, dt):
    """Stored bit pattern -> float32 values (exact for every storage dtype)."""
    if dt == "f32":
        return np.asarray(u, dtype=np.uint32).view(np.float32)
    if dt == "bf16":
        return (np.asarray(u, dtype=np.uint16).astype(np.uint32) << 16).view(np.float32)
    if dt == "f16":
        return np.asarray(u, dtype=np.uint16).view(np.float16).astype(np.float32)
    raise ValueError(dt)


def f32_to_bits(a, dt):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if dt == "f32":
        return a.view(np.uint32)
    if dt == "bf16":
        from oracle.po2_oracle import f32_to_bf16_bits
        return f32_to_bf16_bits(a)
    if dt == "f16":
        return a.astype(np.float16).view(np.uint16)
    raise ValueError(dt)


def same_bits(a_bits, b_bits):
    """Bitwise equality, except that any NaN equals any NaN (payloads are not part of parity)."""
    a = np.asarray(a_bits)
    b = np.asarray(b_bits)
    if a.shape != b.shape:
        return False, -1
    if a.dtype == np.uint32:
        nan = lambda u: (u & 0x7FFFFFFF) > 0x7F800000
    else:
        nan = None
    neq = a != b
    if nan is not None:
        neq &= ~(nan(a) & nan(b))
    idx = np.flatnonzero(neq)
    return idx.size == 0, (int(idx[0]) if idx.size else -1)


def nan_mask(bits, dt):
    v = bits_to_f32(bits, dt)
    return np.isnan(v)


def quantizer_cases():
    """quantizer_golden.npz stores each distinct input once ("input|<i>": flattened, as the differences of
    consecutive bit patterns, which makes the boundary straddlers compress to almost nothing); "cases" names
    every case and "input_of_case" says which input it quantized.  An input has the shape of its output."""
    z = load("quantizer_golden.npz")
    inputs = {}
    for k, i in zip(z["cases"], z["input_of_case"]):
        if i not in inputs:
            d = z[f"input|{i}"]
            inputs[i] = np.cumsum(d, dtype=d.dtype)        # unsigned: wraps modulo 2^bits, undoing the differences
        name, dt, qn, bits = k.split("|")
        y = z[k + "|y"]
        yield str(k), name, dt, qn, int(bits), inputs[i].reshape(y.shape), y
