#!/usr/bin/env python
"""Stage the UNMODIFIED reference (baaivision/Painter) into the git-ignored `oracle/_ref/`, where oracle/ref_loader.py
finds it when $PAINTER_REFERENCE is not set:

    python -m oracle.stage_reference [reference checkout]      # default: $PAINTER_REFERENCE, else DEFAULT_SRC

The reference is pure Python with no setup.py, so there is nothing to compile; this copy is the install step.  Only
the files of the hot path, its two engines, the runtime utilities they import, the data pipeline used by the parity
tests and the SegGPT example images are copied, byte for byte.  Nothing under oracle/_ref is tracked by git or imported
by the product path: it serves the golden generators (oracle/make_golden*.py), the tests that drive the unmodified
reference code and the reference legs of bench.py.
"""
import filecmp
import os
import shutil
import sys

DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
DEFAULT_SRC = "/root/reference"       # the reference checkout looked for when $PAINTER_REFERENCE is not set

FILES = [
    "LICENSE",
    "Painter/models_painter.py",
    "Painter/engine_train.py",
    "Painter/main_train.py",
    "Painter/util",                       # misc, lr_sched, lr_decay, vitdet_utils, masking_generator, ...
    "Painter/data/pairdataset.py",
    "Painter/data/pair_transforms.py",
    "Painter/data/sampler.py",
    "Painter/eval/ade20k_semantic/painter_inference_segm.py",
    "SegGPT/SegGPT_inference/models_seggpt.py",
    "SegGPT/SegGPT_inference/seggpt_engine.py",
    "SegGPT/SegGPT_inference/seggpt_inference.py",
    "SegGPT/SegGPT_inference/util",
    "SegGPT/SegGPT_inference/examples",
]


def source():
    """The reference checkout to stage: $PAINTER_REFERENCE, else DEFAULT_SRC; None when neither holds one."""
    src = os.environ.get("PAINTER_REFERENCE") or DEFAULT_SRC
    return src if os.path.isdir(os.path.join(src, "Painter")) else None


def stage(src_root=None, verbose=True):
    src_root = src_root or source()
    if not src_root or not os.path.isdir(os.path.join(src_root, "Painter")):
        raise RuntimeError(f"reference tree not found at {src_root!r} (pass it or set PAINTER_REFERENCE)")
    n = 0
    for rel in FILES:
        s, d = os.path.join(src_root, rel), os.path.join(DST, rel)
        if os.path.isdir(s):
            for dirpath, _, files in os.walk(s):
                for f in files:
                    if f.endswith((".pyc",)):
                        continue
                    sp = os.path.join(dirpath, f)
                    dp = os.path.join(d, os.path.relpath(sp, s))
                    n += _copy(sp, dp)
        else:
            n += _copy(s, d)
    if verbose:
        print(f"staged reference -> {DST} ({n} files copied)")
    return DST


def _copy(s, d):
    os.makedirs(os.path.dirname(d), exist_ok=True)
    if os.path.exists(d) and filecmp.cmp(s, d, shallow=False):
        return 0
    shutil.copyfile(s, d)
    return 1


if __name__ == "__main__":
    stage(sys.argv[1] if len(sys.argv) > 1 else None)
