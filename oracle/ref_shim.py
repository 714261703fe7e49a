"""ORACLE (test infrastructure) — import the UNMODIFIED reference hooks and drivers from the reference tree.

Only usable where the reference tree exists (TOKENFLOW_REFERENCE_DIR); used by `oracle/gen_golden.py`
to produce `tests/golden/`, which the tests compare against.  Nothing is copied: the reference files
are imported from where they lie.

Why a shim is needed (SURVEY.md §8c): reference util.py:8 imports torchvision.io.read_video /
write_video (removed in torchvision 0.26) and util.py:14-15 import kornia (not installed).
Neither is used on the hot path, so inert stand-ins are registered before the import.
"""
from __future__ import annotations

import importlib
import os
import sys
import types

REFERENCE_DIR = os.environ.get("TOKENFLOW_REFERENCE_DIR", "/root/reference")


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_DIR, "tokenflow_utils.py"))


def load_reference():
    """Returns (ref_tokenflow_utils, ref_util) modules, imported under private names so they never
    shadow this repo's drop-in `tokenflow_utils` / `util`."""
    if not reference_available():
        raise FileNotFoundError(f"reference tree not found at {REFERENCE_DIR}")
    if "_ref_tokenflow_utils" in sys.modules:
        return sys.modules["_ref_tokenflow_utils"], sys.modules["_ref_util"]

    import torchvision.io as tvio

    def _absent(*a, **k):
        raise RuntimeError("video I/O is not available in this environment")

    for name in ("read_video", "write_video"):
        if not hasattr(tvio, name):
            setattr(tvio, name, _absent)
    stubs = {}
    for name, attrs in (("kornia", ()), ("kornia.geometry", ()), ("kornia.geometry.transform", ("remap",)),
                        ("kornia.utils", ()), ("kornia.utils.grid", ("create_meshgrid",))):
        if name not in sys.modules:
            m = types.ModuleType(name)
            for a in attrs:
                setattr(m, a, _absent)
            sys.modules[name] = m
            stubs[name] = m

    def _load(private_name: str, filename: str, aliases=()):
        spec = importlib.util.spec_from_file_location(private_name, os.path.join(REFERENCE_DIR, filename))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[private_name] = mod
        saved = {a: sys.modules.get(a) for a in aliases}
        for a in aliases:
            sys.modules[a] = mod
        return mod, spec, saved

    # reference util.py first; reference tokenflow_utils.py does `from util import ...`
    ref_util, spec_u, _ = _load("_ref_util", "util.py")
    spec_u.loader.exec_module(ref_util)
    saved_util = sys.modules.get("util")
    sys.modules["util"] = ref_util
    try:
        ref_tf, spec_t, _ = _load("_ref_tokenflow_utils", "tokenflow_utils.py")
        spec_t.loader.exec_module(ref_tf)
    finally:
        if saved_util is not None:
            sys.modules["util"] = saved_util
        else:
            del sys.modules["util"]
    return ref_tf, ref_util


def load_driver(filename: str, scheduler_cls):
    """Import a reference driver (run_tokenflow_pnp.py / run_tokenflow_sdedit.py) with its `tokenflow_utils`
    and `util` imports resolving to this repo's top-level drop-in modules.  `diffusers` is not installed: a
    stub supplies `scheduler_cls` as its DDIMScheduler and an empty StableDiffusionPipeline (the driver's
    __init__, which loads Stable Diffusion, is never run)."""
    if not reference_available():
        raise FileNotFoundError(f"reference tree not found at {REFERENCE_DIR}")
    import tokenflow_utils as dropin_tf
    import util as dropin_util
    stub = types.ModuleType("diffusers")
    stub.DDIMScheduler = scheduler_cls
    stub.StableDiffusionPipeline = type("StableDiffusionPipeline", (), {})
    saved = {k: sys.modules.get(k) for k in ("diffusers", "tokenflow_utils", "util")}
    sys.modules.update({"diffusers": stub, "tokenflow_utils": dropin_tf, "util": dropin_util})
    try:
        name = "_ref_driver_" + filename.replace(".py", "")
        spec = importlib.util.spec_from_file_location(name, os.path.join(REFERENCE_DIR, filename))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)             # `if __name__ == '__main__'` does not fire
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return mod
