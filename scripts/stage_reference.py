#!/usr/bin/env python
"""Stage the reference's own Python sources for the hot path under the git-ignored ``baseline/_ref/`` so that a copy
of this working tree carries them to a machine without the original project's checkout.

    VADC_REFERENCE_ROOT=<checkout of the original project> python scripts/stage_reference.py   # no-op without it

The reference is not pip-installable (no setup.py / pyproject, SURVEY.md 2), so "installing" it is a copy of the
package directories the path imports: model/ (cluster, Memory, backbone + the encoder / decoder files backbone
imports), loss_tool/, misc/, utils/, tool/.  Nothing staged here is part of the product or of the git history:
``baseline/_ref`` is used by ``bench.py --impl reference`` (the reference's own classes timed on the host cores),
by the ``gpu_reference`` leg of bench.py (the same classes on CUDA tensors — SURVEY 2.2's "real bar") and by the
model-level drop-in test (tests/test_gpu_dropin_model.py)."""
import hashlib
import json
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("VADC_REFERENCE_ROOT", "")
DST = os.path.join(ROOT, "baseline", "_ref")
PACKAGES = ["model", "loss_tool", "misc", "utils", "tool"]


def stage(verbose=True):
    if not REF or not os.path.isdir(os.path.join(REF, "model")):
        if verbose:
            print(f"stage_reference: no reference checkout at VADC_REFERENCE_ROOT={REF!r}; keeping {DST} as it is")
        return False
    manifest = {}
    for pkg in PACKAGES:
        for dirpath, dirnames, filenames in os.walk(os.path.join(REF, pkg)):
            dirnames[:] = [d for d in dirnames if d != "__pycache__"]
            for fn in filenames:
                if not fn.endswith(".py"):
                    continue
                src = os.path.join(dirpath, fn)
                rel = os.path.relpath(src, REF)
                dst = os.path.join(DST, rel)
                os.makedirs(os.path.dirname(dst), exist_ok=True)
                shutil.copyfile(src, dst)
                with open(src, "rb") as fh:
                    manifest[rel] = hashlib.sha256(fh.read()).hexdigest()
    with open(os.path.join(DST, "MANIFEST.json"), "w") as fh:
        json.dump({"source": REF, "files": manifest}, fh, indent=1, sort_keys=True)
    if verbose:
        print(f"stage_reference: {len(manifest)} files -> {DST}")
    return True


if __name__ == "__main__":
    stage()
    sys.exit(0)
