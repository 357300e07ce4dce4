"""TEST INFRASTRUCTURE: import the UNMODIFIED reference modules through the shim packages in oracle/shims
(timm 0.3.2 symbols, import-only detectron2/fairscale/fvcore, torch._six).

The reference tree is looked up at $PAINTER_REFERENCE, then at the staged byte-for-byte copy under oracle/_ref/
(oracle/stage_reference.py; git-ignored).  Nothing in the product path (painter_b200/*) imports this file: only the
golden generators, the tests that drive the unmodified reference code, the `--impl reference` / cpu_baseline legs of
bench.py and scripts under scripts/ do.
"""
import importlib
import importlib.util
import os
import sys
import types

_HERE = os.path.dirname(os.path.abspath(__file__))
_SHIMS = os.path.join(_HERE, "shims")
_STAGED = os.path.join(_HERE, "_ref")


def _find_root():
    for cand in (os.environ.get("PAINTER_REFERENCE"), _STAGED):
        if cand and os.path.isdir(os.path.join(cand, "Painter")):
            return cand
    return _STAGED


REF_ROOT = _find_root()


def available():
    return os.path.isdir(os.path.join(REF_ROOT, "Painter"))


def _install_shims():
    if _SHIMS not in sys.path:
        sys.path.insert(0, _SHIMS)
    if "torch._six" not in sys.modules:  # Painter/util/misc.py:22
        import math
        m = types.ModuleType("torch._six")
        m.inf = math.inf
        sys.modules["torch._six"] = m


def _load(name, path, pkg_dir):
    """Load `path` as module `name` with pkg_dir temporarily first on sys.path (for `util.*`)."""
    _install_shims()
    saved = {k: v for k, v in sys.modules.items() if k == "util" or k.startswith("util.")}
    for k in saved:
        del sys.modules[k]
    sys.path.insert(0, pkg_dir)
    try:
        spec = importlib.util.spec_from_file_location(name, path)
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
    finally:
        sys.path.remove(pkg_dir)
        for k in [k for k in sys.modules if k == "util" or k.startswith("util.")]:
            sys.modules["_ref_" + name + "." + k] = sys.modules.pop(k)
        sys.modules.update(saved)
    return mod


_cache = {}


def models_painter():
    if "p" not in _cache:
        d = os.path.join(REF_ROOT, "Painter")
        _cache["p"] = _load("ref_models_painter", os.path.join(d, "models_painter.py"), d)
    return _cache["p"]


def models_seggpt():
    if "s" not in _cache:
        d = os.path.join(REF_ROOT, "SegGPT", "SegGPT_inference")
        _cache["s"] = _load("ref_models_seggpt", os.path.join(d, "models_seggpt.py"), d)
    return _cache["s"]


def masking_generator():
    if "m" not in _cache:
        d = os.path.join(REF_ROOT, "Painter")
        _cache["m"] = _load("ref_masking_generator", os.path.join(d, "util", "masking_generator.py"), d)
    return _cache["m"]


def engine_train():
    """Painter/engine_train.py (train_one_epoch, evaluate_pt) with its own `util.misc` / `util.lr_sched`."""
    if "e" not in _cache:
        d = os.path.join(REF_ROOT, "Painter")
        _cache["e"] = _load("ref_engine_train", os.path.join(d, "engine_train.py"), d)
    return _cache["e"]


def misc():
    """Painter/util/misc.py as imported by engine_train (NativeScalerWithGradNormCount, save_model, ...)."""
    engine_train()
    return sys.modules["_ref_ref_engine_train.util.misc"]


def lr_decay():
    if "ld" not in _cache:
        d = os.path.join(REF_ROOT, "Painter")
        _cache["ld"] = _load("ref_lr_decay", os.path.join(d, "util", "lr_decay.py"), d)
    return _cache["ld"]


def seggpt_engine():
    """SegGPT/SegGPT_inference/seggpt_engine.py (run_one_image, inference_image, inference_video)."""
    if "se" not in _cache:
        d = os.path.join(REF_ROOT, "SegGPT", "SegGPT_inference")
        _cache["se"] = _load("ref_seggpt_engine", os.path.join(d, "seggpt_engine.py"), d)
    return _cache["se"]


def painter_inference_segm():
    """Painter/eval/ade20k_semantic/painter_inference_segm.py (run_one_image :67-93)."""
    if "pi" not in _cache:
        d = os.path.join(REF_ROOT, "Painter")
        # the script imports matplotlib.pyplot (unused by run_one_image; absent from this image) and its sibling
        # `models_painter` by bare name: both are provided for the duration of the import only
        injected = []
        try:
            import matplotlib.pyplot  # noqa: F401
        except Exception:
            for n in ("matplotlib", "matplotlib.pyplot"):
                sys.modules[n] = types.ModuleType(n)
                injected.append(n)
        had_mp = sys.modules.get("models_painter")
        sys.modules["models_painter"] = models_painter()
        try:
            _cache["pi"] = _load("ref_painter_inference_segm",
                                 os.path.join(d, "eval", "ade20k_semantic", "painter_inference_segm.py"), d)
        finally:
            for n in injected:
                sys.modules.pop(n, None)
            if had_mp is None:
                sys.modules.pop("models_painter", None)
            else:
                sys.modules["models_painter"] = had_mp
    return _cache["pi"]


def pairdataset():
    if "pd" not in _cache:
        d = os.path.join(REF_ROOT, "Painter")
        _cache["pd"] = _load("ref_pairdataset", os.path.join(d, "data", "pairdataset.py"), d)
    return _cache["pd"]


def examples_dir():
    return os.path.join(REF_ROOT, "SegGPT", "SegGPT_inference", "examples")
