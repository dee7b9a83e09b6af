"""Imports the REAL reference modules from a checkout of endiqq/Multi-Feature-ViT named by the MFVIT_REFERENCE
environment variable (the repository does not contain it).  Used by oracle/gen_golden.py to produce tests/golden/*.pt.
TEST INFRASTRUCTURE ONLY."""
import importlib
import os
import sys
import types

REFERENCE = os.environ.get("MFVIT_REFERENCE", "")
REF_ROOT = os.path.join(REFERENCE, "moco_pretraining", "moco") if REFERENCE else ""
FUS_MODULE = ("model.crossvit_2vits_2additionaloutputs_changenormlayer_location_removeextralclayer_"
              "changemodelinputlocation_std002_sum")
BLD_MODULE = "moco.builder_vit_mocov3structure_mocov2loss"


def available():
    return bool(REF_ROOT) and os.path.isdir(REF_ROOT)


def _install_timm_shim():
    """FUS:9 imports DropPath, to_2tuple, trunc_normal_ from timm.models.layers; only trunc_normal_ is used (FUS:119)."""
    import torch
    if "timm" in sys.modules:
        return
    timm = types.ModuleType("timm")
    models = types.ModuleType("timm.models")
    layers = types.ModuleType("timm.models.layers")
    layers.trunc_normal_ = torch.nn.init.trunc_normal_
    layers.to_2tuple = lambda x: (x, x) if not isinstance(x, tuple) else x
    layers.DropPath = torch.nn.Identity
    timm.models, models.layers = models, layers
    sys.modules.update({"timm": timm, "timm.models": models, "timm.models.layers": layers})


class _RefPath:
    """Temporarily puts the reference package root first on sys.path and hides same-named drop-in modules."""

    def __enter__(self):
        self.saved = {k: v for k, v in sys.modules.items() if k.split(".")[0] in ("model", "moco")}
        for k in self.saved:
            del sys.modules[k]
        # the reference's moco/ has no __init__.py (a namespace package): a regular package of the same name anywhere
        # on sys.path - the drop-in's - would win, so the drop-in directory is hidden for the duration of the import
        self.saved_path = list(sys.path)
        sys.path[:] = [REF_ROOT] + [p for p in sys.path if os.path.basename(os.path.normpath(p)) != "dropin"]
        return self

    def __exit__(self, *exc):
        sys.path[:] = self.saved_path
        self.loaded = {k: v for k, v in sys.modules.items() if k.split(".")[0] in ("model", "moco")}
        for k in self.loaded:
            del sys.modules[k]
        sys.modules.update(self.saved)


def load_reference():
    """Returns (module_py, fus_py, bld_py): the real MOD, FUS and BLD modules."""
    if not available():
        raise RuntimeError("reference tree not found: set MFVIT_REFERENCE to a checkout of endiqq/Multi-Feature-ViT")
    _install_timm_shim()
    with _RefPath():
        mod = importlib.import_module("model.module")
        fus = importlib.import_module(FUS_MODULE)
        bld = importlib.import_module(BLD_MODULE)
    return mod, fus, bld
