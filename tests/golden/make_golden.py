"""Generate golden input/output vectors from the UNMODIFIED reference (run in the build container).

    PO2_REFERENCE=<checkout> python tests/golden/make_golden.py      # writes tests/golden/*.npz

The reference is Python and cannot travel to the GPU box, so its outputs on seeded inputs are
committed as fixtures.  Tensors are stored as raw bit patterns (uint32 for fp32, uint16 for
bf16/fp16) so that NaN payloads, signed zeros and subnormals survive exactly.
"""
import os
import sys

import numpy as np
import torch

REF = os.environ.get("PO2_REFERENCE") or sys.exit("make_golden.py: set PO2_REFERENCE to a checkout of the reference")
sys.path.insert(0, REF)
from utils.quantizers import (PowerOfTwoPlusQuantizer, PowerOfTwoQuantizer,  # noqa: E402
                              LinearPowerOfTwoQuantizer, LinearPowerOfTwoPlusQuantizer,
                              quantize_model)
from models.model import get_model  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
TD = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
Q = {"po2": PowerOfTwoQuantizer, "po2+": PowerOfTwoPlusQuantizer}


def bits_of(t: torch.Tensor) -> np.ndarray:
    if t.dtype == torch.float32:
        return t.contiguous().view(torch.int32).numpy().view(np.uint32).copy()
    return t.contiguous().view(torch.int16).numpy().view(np.uint16).copy()


def f32_from_bits(u):
    return torch.from_numpy(np.asarray(u, dtype=np.uint32).view(np.int32).copy()).view(torch.float32)


def boundary_inputs(plus: bool, scale: float) -> torch.Tensor:
    """fp32 values straddling every rounding boundary of round(log2(.)) for v in [2^-128, 1)."""
    centre = 0x400000 if plus else 0x3504F3
    out = []
    for e in range(-126, 0):
        m = np.arange(centre - 40, centre + 41, dtype=np.int64)
        out.append((((e + 127) << 23) | m).astype(np.uint32))
    # subnormal v (only reachable at bits=8): mantissa threshold without the implicit bit
    sub_c = int(round((1.5 if plus else 2 ** 0.5) * 2 ** 22))
    out.append(np.arange(sub_c - 40, sub_c + 41, dtype=np.uint32))
    v = f32_from_bits(np.concatenate(out))
    s = torch.tensor(scale, dtype=torch.float32)
    x = v * s                       # fl(v*s); the division below re-derives its own v
    # neighbours, so that fl(x/s) lands on both sides of each boundary whatever s is
    xb = x.view(torch.int32)
    x = torch.cat([torch.clamp(xb + d, min=0).view(torch.float32) for d in (-2, -1, 0, 1, 2)])
    x = x[x <= s]
    sgn = torch.where(torch.arange(x.numel()) % 3 == 0, -1.0, 1.0)
    x = torch.cat([x * sgn, s.reshape(1)])       # plant the max so that scale == s
    assert torch.max(torch.abs(x)).item() == s.item()
    return x


def save_quantizer_cases(path, cases):
    """{"<case>|x": bits, "<case>|y": bits} -> the layout tests/golden_util.quantizer_cases() reads: each distinct
    input once, flattened and stored as differences of consecutive bit patterns (the file stays under 1 MB)."""
    keys = sorted(k[:-2] for k in cases if k.endswith("|x"))
    inputs, index, out = {}, [], {}
    for k in keys:
        x = cases[k + "|x"]
        i = inputs.setdefault((x.dtype.str, x.shape, x.tobytes()), len(inputs))
        if f"input|{i}" not in out:
            f = x.ravel()
            out[f"input|{i}"] = np.diff(f, prepend=f.dtype.type(0)).astype(f.dtype)
        index.append(i)
        out[k + "|y"] = cases[k + "|y"]
    np.savez_compressed(path, cases=np.array(keys), input_of_case=np.array(index, dtype=np.int32), **out)


def main():
    torch.manual_seed(1234)
    g = torch.Generator().manual_seed(1234)
    cases = {}
    base = {
        "randn": torch.randn(4099, generator=g),
        "heavy": torch.randn(4099, generator=g) ** 3,
        "weightlike": torch.randn(64, 16, 3, 3, generator=g) * 0.05,
        "tiny_scale": torch.randn(1025, generator=g) * 1e-39,
        "huge_scale": torch.randn(1025, generator=g) * 1e37,
        "edge": torch.tensor([1.0, -0.5, 0.0, -0.0, 1e-30, 0.75, 0.375, 0.1875, -0.75, 1.5 * 2 ** -7,
                              2 ** -6.5, 2 ** -7.5, 2 ** -8, 1e-45, -1e-45, 2.0 ** -126, 0.70710678,
                              0.70710677, 0.7071068, 0.35355338, 0.35355339, 3e-39, 2.0 ** -127]),
        "single": torch.tensor([-3.25]),
        "with_inf": torch.tensor([1.0, float("inf"), 0.0, -2.0, float("-inf"), 1e-3]),
        "with_nan": torch.tensor([1.0, float("nan"), 0.0, -2.0]),
        "all_zero": torch.zeros(7),
    }
    for name, x in base.items():
        for dt in ("f32", "bf16", "f16"):
            xd = x.to(TD[dt])
            for qn, qc in Q.items():
                for bits in (2, 3, 4, 5, 8):
                    if dt == "f16" and name in ("huge_scale",):
                        continue
                    y = qc.forward(None, xd, bits=bits)
                    key = f"{name}|{dt}|{qn}|{bits}"
                    cases[key + "|x"] = bits_of(xd)
                    cases[key + "|y"] = bits_of(y)
    # boundary straddlers, fp32 only (the libm-sensitive vectors)
    for qn, qc in Q.items():
        for si, s in enumerate((1.0, 1.337, 0.0517, 1.4142135, 1.3333334, 3e-39, 7.7e30)):
            x = boundary_inputs(qn == "po2+", s)
            for bits in (4, 8):
                y = qc.forward(None, x, bits=bits)
                key = f"boundary{si}|f32|{qn}|{bits}"
                cases[key + "|x"] = bits_of(x)
                cases[key + "|y"] = bits_of(y)
    # fsr != 1 (accepted by the signature, utils/quantizers.py:21, never used by a caller)
    x = base["randn"]
    for qn, qc in Q.items():
        for fsr in (0, 2):
            y = qc.forward(None, x, bits=4, fsr=fsr)
            cases[f"fsr{fsr}|f32|{qn}|4|x"] = bits_of(x)
            cases[f"fsr{fsr}|f32|{qn}|4|y"] = bits_of(y)
    save_quantizer_cases(os.path.join(HERE, "quantizer_golden.npz"), cases)
    print("quantizer cases:", len(cases) // 2)

    # statistical known answer (SURVEY.md section 4): po2 -> po2+ MSE change on randn(2^20)
    xs = torch.randn(2 ** 20, generator=torch.Generator().manual_seed(1234))
    ka = {}
    for bits in (2, 3, 4, 8):
        for qn, qc in Q.items():
            y = qc.forward(None, xs, bits=bits)
            ka[f"mse|{qn}|{bits}"] = np.float64(torch.mean((y - xs).double() ** 2).item())
    # quantize_model known answers on the seeded ResNet-20 (utils/quantizers.py:139-153)
    for qn, qc in Q.items():
        for bits in (3, 4):
            torch.manual_seed(8)
            m = get_model("resnet20", 10, None, bits, (32, 32))
            ka[f"resnet20_ptq_mse|{qn}|{bits}"] = np.float64(quantize_model(m, qc, bits))
    # lin / lin+ (scope row f1) on a conv-weight-shaped tensor
    w = torch.randn(32, 16, 3, 3, generator=torch.Generator().manual_seed(5)) * 0.1
    lin = {"w": w.numpy()}
    for nm, qc in (("lin", LinearPowerOfTwoQuantizer), ("lin+", LinearPowerOfTwoPlusQuantizer)):
        for bits in (3, 4):
            lin[f"{nm}|{bits}"] = qc.forward(None, w, bits=bits).numpy()
    np.savez_compressed(os.path.join(HERE, "known_answers.npz"), **ka)
    np.savez_compressed(os.path.join(HERE, "lin_golden.npz"), **lin)
    print({k: float(v) for k, v in ka.items()})


if __name__ == "__main__":
    main()
