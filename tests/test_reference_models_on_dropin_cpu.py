"""The reference's OWN model files (models/resnet.py, mobilenet.py, mobile_vit.py) build and run,
unchanged, on top of this repo's drop-in `QuantizedConv2d` / `utils.quantizers`, and this repo's
workload graphs are parameter-for-parameter the same networks.  Those tests need a checkout of the
reference, which the repository does not contain ($PO2_REFERENCE, or staged into baseline/_ref), and skip
without one; the structure the reference's models were probed to have is stored in
tests/golden/reference_model_structure.json and checked on every run."""
import copy
import importlib
import json
import os
import sys

import pytest
import torch

from workloads.reference_files import find_reference

REF = find_reference()
needs_checkout = pytest.mark.skipif(REF is None, reason="no reference checkout ($PO2_REFERENCE or baseline/_ref)")


@pytest.fixture
def ref_models_on_dropin():
    """Import the reference's `models` package with models.quantized_conv / utils.quantizers replaced
    by the drop-in shims (what INTEGRATION.md tells a user to do)."""
    import drop_in.models.quantized_conv as qc
    import drop_in.utils.quantizers as uq
    saved = {k: sys.modules.get(k) for k in list(sys.modules) if k == "models" or k.startswith("models.") or k == "utils" or k.startswith("utils.")}
    for k in saved:
        sys.modules.pop(k, None)
    sys.path.insert(0, REF)
    try:
        import models  # noqa: F401  (reference package)
        sys.modules["models.quantized_conv"] = qc
        import utils  # noqa: F401
        sys.modules["utils.quantizers"] = uq
        model_mod = importlib.import_module("models.model")
        yield model_mod
    finally:
        sys.path.remove(REF)
        for k in [k for k in sys.modules if k == "models" or k.startswith("models.") or k == "utils" or k.startswith("utils.")]:
            sys.modules.pop(k, None)
        for k, v in saved.items():
            if v is not None:
                sys.modules[k] = v


@needs_checkout
@pytest.mark.parametrize("name", ["resnet20", "resnet56", "mobilenet", "mobilevit"])
def test_reference_model_files_run_on_dropin_and_match_workloads(ref_models_on_dropin, name):
    import po2_quantization_b200 as P
    from workloads import mobilenet_v2_cifar, mobilevit_xs, resnet_cifar
    torch.manual_seed(8)
    ref = ref_models_on_dropin.get_model(name, 10, None, 4, (32, 32))
    qconvs = [m for m in ref.modules() if isinstance(m, P.QuantizedConv2d)]
    assert len(qconvs) == {"resnet20": 20, "resnet56": 56, "mobilenet": 50, "mobilevit": 33}[name]
    mine = {"resnet20": lambda: resnet_cifar(20), "resnet56": lambda: resnet_cifar(56),
            "mobilenet": lambda: mobilenet_v2_cifar(), "mobilevit": lambda: mobilevit_xs((32, 32), 10, (1, 1), None, 4)}[name]()
    sr, sm = ref.state_dict(), mine.state_dict()
    assert list(sr) == list(sm) and all(sr[k].shape == sm[k].shape for k in sr)
    mine.load_state_dict(sr, strict=True)
    ref.eval(); mine.eval()
    x = torch.randn(2, 3, 32, 32)
    with torch.no_grad():
        assert torch.equal(ref(x), mine(x))           # quantize_fn=None on CPU: nn.Conv2d's own path
    c = copy.deepcopy(ref)                            # test.py:120
    assert list(c.state_dict()) == list(sr)
    err, numel = ref.get_quantization_error()         # models/*.py walkers call QuantizedConv2d.get_quantization_error
    assert err == 0 and numel > 0


@needs_checkout
def test_reference_qat_model_builds_with_dropin_quantizer(ref_models_on_dropin):
    import po2_quantization_b200 as P
    m = ref_models_on_dropin.get_model("resnet20", 10, P.PowerOfTwoPlusQuantizer, 4, (32, 32))
    q = [mm for mm in m.modules() if isinstance(mm, P.QuantizedConv2d)]
    assert all(mm.quantize_fn is P.PowerOfTwoPlusQuantizer and mm.bits == 4 for mm in q)
    with pytest.raises(Exception) as ei:              # CPU tensors: loud failure, no silent fallback
        m(torch.randn(1, 3, 32, 32))
    assert "no CPU fallback" in str(ei.value)


def _workload(name):
    from workloads import mobilenet_v2_cifar, mobilevit_xs, resnet_cifar
    return {"resnet20": lambda: resnet_cifar(20), "resnet56": lambda: resnet_cifar(56),
            "mobilenet": lambda: mobilenet_v2_cifar(), "mobilevit": lambda: mobilevit_xs((32, 32), 10, (1, 1), None, 4)}[name]()


@pytest.mark.parametrize("name", ["resnet20", "resnet56", "mobilenet", "mobilevit"])
def test_workload_graphs_have_the_reference_model_structure(name):
    """The networks the drop-in classes run against what the unmodified reference models were probed to be
    (tests/golden/reference_model_structure.json): every QuantizedConv2d's shape, stride and feature-map size
    (forward hooks on one 3x32x32 image), MACs per image, norm layers and parameter count."""
    import po2_quantization_b200 as P
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_model_structure.json")) as f:
        want = json.load(f)["models"][name]
    torch.manual_seed(8)
    model = _workload(name).eval()
    rows = []
    hook = lambda m, inp, out: rows.append((m.in_channels, m.out_channels, m.kernel_size[0], m.stride[0], m.padding[0],
                                            m.groups, inp[0].shape[-1], out.shape[-1], out.shape[-2] * out.shape[-1] * m.weight.numel()))
    handles = [m.register_forward_hook(hook) for m in model.modules() if isinstance(m, P.QuantizedConv2d)]
    with torch.no_grad():
        model(torch.randn(1, 3, 32, 32))
    for h in handles:
        h.remove()
    assert len(rows) == want["quantized_convs"]
    assert sum(1 for r in rows if r[5] > 1) == want["depthwise"]
    assert sum(1 for r in rows if r[2] == 1) == want["pointwise"]
    assert round(sum(r[8] for r in rows) / 1e6, 2) == want["qconv_mmac_per_image"]
    if "depthwise_mmac_per_image" in want:
        assert round(sum(r[8] for r in rows if r[5] > 1) / 1e6, 2) == want["depthwise_mmac_per_image"]
    if "layers" in want:
        shapes = {}
        for c, k, ks, s, p, _, h, q, _ in rows:
            shapes[(c, k, ks, s, p, h, q)] = shapes.get((c, k, ks, s, p, h, q), 0) + 1
        assert shapes == {tuple(r[:7]): r[7] for r in want["layers"]}
    norms = sum(1 for m in model.modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm))
    assert norms == want["norm_layers"]
    n_params = sum(p.numel() for p in model.parameters())
    if "parameters" in want:
        assert n_params == want["parameters"]
    if "parameter_mbytes" in want:
        assert round(n_params * 4 / 1e6, 1) == want["parameter_mbytes"]
