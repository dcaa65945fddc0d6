"""Import the reference's OWN model files, unmodified, from a checkout named by $PO2_REFERENCE or staged
into baseline/_ref/ by baseline/stage_reference.py.  The repository does not contain them.

Two variants of the same files:
  * ``load("dropin")`` -- `models.quantized_conv` and `utils.quantizers` replaced by this repo's drop-in
    shims (drop_in/, what INTEGRATION.md tells a user to do): the reference's ResNet / MobileNetV2 /
    MobileViT definitions then run on the sm_100a kernels without a single edit;
  * ``load("stock")``  -- everything from the reference, i.e. its torch-op quantizers and nn.Conv2d's
    convolution: the reference itself, runnable on CPU (the baseline arm) or on CUDA (the GPU oracle).

The reference uses absolute imports (`from models.quantized_conv import ...`), so each variant is
imported with `models` / `utils` temporarily bound in sys.modules and unbound again afterwards; the
returned namespace keeps the module objects alive.
"""
import importlib
import os
import sys
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_cache = {}


def find_reference():
    for p in (os.environ.get("PO2_REFERENCE"), os.path.join(ROOT, "baseline", "_ref")):
        if p and os.path.isfile(os.path.join(p, "models", "model.py")) and os.path.isfile(os.path.join(p, "utils", "quantizers.py")):
            return p
    return None


def _ours(name):
    return name == "models" or name.startswith("models.") or name == "utils" or name.startswith("utils.")


def load(variant: str = "dropin"):
    """-> namespace(get_model, quantizers, QuantizedConv2d, MobileViT, path, variant), or None when no
    reference checkout is available."""
    if variant not in ("dropin", "stock"):
        raise ValueError("variant must be 'dropin' or 'stock'")
    if variant in _cache:
        return _cache[variant]
    ref = find_reference()
    if ref is None:
        return None
    saved = {k: v for k, v in sys.modules.items() if _ours(k)}
    for k in saved:
        del sys.modules[k]
    sys.path.insert(0, ref)
    try:
        importlib.import_module("models")
        importlib.import_module("utils")
        if variant == "dropin":
            import drop_in.models.quantized_conv as qc
            import drop_in.utils.quantizers as uq
            sys.modules["models.quantized_conv"] = qc
            sys.modules["utils.quantizers"] = uq
        else:
            qc = importlib.import_module("models.quantized_conv")
            uq = importlib.import_module("utils.quantizers")
        model_mod = importlib.import_module("models.model")
        vit_mod = importlib.import_module("models.mobile_vit")
        ns = SimpleNamespace(get_model=model_mod.get_model, quantizers=uq, QuantizedConv2d=qc.QuantizedConv2d,
                             MobileViT=vit_mod.MobileViT, path=ref, variant=variant)
    finally:
        sys.path.remove(ref)
        for k in [k for k in sys.modules if _ours(k)]:
            del sys.modules[k]
        sys.modules.update(saved)
    _cache[variant] = ns
    return ns


def mobilevit_224(ns, num_classes=1000, quantize_fn=None, bits=8):
    """BASELINE.json configs[3] at 224x224: the reference's factory cannot build a working 224x224 model
    (SURVEY.md section 5), so the class is constructed directly with patch_size (1,1) -- section 8d (i)."""
    return ns.MobileViT(image_size=(224, 224), dims=(96, 120, 144), channels=(16, 32, 48, 48, 64, 64, 80, 80, 96, 96, 384),
                        num_classes=num_classes, patch_size=(1, 1), quantize_fn=quantize_fn, bits=bits)
