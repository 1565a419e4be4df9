"""Import the UNMODIFIED reference modules from the original project's source tree.

TEST INFRASTRUCTURE ONLY.  The tree is not part of this repository: point MWA_REFERENCE_ROOT at a
checkout of it to enable the tests that compare against it live; without it `available()` is False
and they skip (tests/golden holds stored outputs of the same modules).  No reference source is
copied -- the modules are executed from where they lie, through the stand-in packages under shims/.
"""
from __future__ import annotations

import importlib
import os
import sys

REFERENCE_ROOT = os.environ.get("MWA_REFERENCE_ROOT", "")
_SHIMS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "shims")


def available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "layers", "masked_win_attention.py"))


class _RefModules:
    def __init__(self):
        self.masked = importlib.import_module("layers.masked_win_attention")
        self.unmasked = importlib.import_module("layers.win_attention")
        self.gdn = importlib.import_module("layers.GDN")
        self.wrapper = importlib.import_module("layers.Masked_Attention")
        self.supply = importlib.import_module("layers.SupplyMask")

    def script(self, which: str = "trainRGB"):
        """the training / evaluation script as a module (its argparse runs in main() only); its module-level `device`
        is the hard-coded 'cuda:0' (trainRGB.py:31) -- set to 'cpu' so that `constraint` runs in this container"""
        argv, sys.argv = sys.argv, [which]
        try:
            mod = importlib.import_module(which)
        finally:
            sys.argv = argv
        mod.device = "cpu"
        return mod

    def model(self, which: str):
        """'rgb' -> models.AutoEncoderRGB_Journal, 'mask' -> models.AutoEncoderMask_Journal."""
        name = {"rgb": "models.AutoEncoderRGB_Journal", "mask": "models.AutoEncoderMask_Journal"}[which]
        return importlib.import_module(name)


_cached = None


def load() -> _RefModules:
    """Put shims + reference on sys.path (the tree is read-only: no bytecode) and import."""
    global _cached
    if _cached is not None:
        return _cached
    if not available():
        raise RuntimeError(f"reference tree not found at MWA_REFERENCE_ROOT={REFERENCE_ROOT!r}")
    sys.dont_write_bytecode = True
    for p in (REFERENCE_ROOT, _SHIMS):
        if p not in sys.path:
            sys.path.insert(0, p)
    for name in ("layers", "models"):
        mod = sys.modules.get(name)
        if mod is not None and not str(getattr(mod, "__path__", [""])[0]).startswith(REFERENCE_ROOT):
            raise RuntimeError(f"a different '{name}' package is already imported")
    _cached = _RefModules()
    return _cached
