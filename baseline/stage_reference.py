"""Stage the reference's model files next to the repo so that they can travel to the GPU box.

    python baseline/stage_reference.py [CHECKOUT]  # CHECKOUT (default $PO2_REFERENCE) -> baseline/_ref/

The reference (mschoenb97/po2_quantization) is a flat script repo without setup.py / pyproject, so
`pip install --target baseline/_ref /root/reference` has nothing to install; what the GPU-side tests and
`bench.py` need from it are the files that CALL the hot path, unmodified: `models/*.py` (ResNet,
MobileNetV2, MobileViT, the factory, the reference QuantizedConv2d) and `utils/quantizers.py`.  They are
copied verbatim into baseline/_ref/ (git-ignored: reference sources never enter this repo's history;
not gpurun-ignored: the directory ships with the snapshot like the built .so).  Nothing is edited.
`__graft_entry__.build()` runs this; without a checkout it stages nothing.
"""
import filecmp
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "baseline", "_ref")
FILES = ["models/__init__.py", "models/model.py", "models/resnet.py", "models/mobilenet.py", "models/mobile_vit.py",
         "models/quantized_conv.py", "utils/__init__.py", "utils/quantizers.py"]


def stage(src: str = None, verbose: bool = True) -> bool:
    src = src or os.environ.get("PO2_REFERENCE")
    if not src or not os.path.isdir(os.path.join(src, "models")):
        if verbose:
            print(f"[stage_reference] no reference checkout ({src or '$PO2_REFERENCE unset'}): nothing staged")
        return False
    n = 0
    for rel in FILES:
        s, d = os.path.join(src, rel), os.path.join(DST, rel)
        os.makedirs(os.path.dirname(d), exist_ok=True)
        if not (os.path.exists(d) and filecmp.cmp(s, d, shallow=False)):
            shutil.copyfile(s, d)
            n += 1
    if verbose:
        print(f"[stage_reference] {len(FILES)} reference files in {DST} ({n} copied)")
    return True


if __name__ == "__main__":
    stage(sys.argv[1] if len(sys.argv) > 1 else None)
