"""Import the reference's own hot-path modules in place from a lightly-train source tree ($LIGHTLY_TRAIN_SRC, the
checkout's `src` directory).

`import lightly_train` itself fails here (its __init__ pulls pytorch_lightning / albumentations / omegaconf /
lightly, none installed).  Registering an empty namespace package whose __path__ is the reference source
directory skips that __init__, and a 5-line stub of lightning_utilities.core.imports.RequirementCache (used at
vision_transformer.py:24,43) is enough for the arithmetic modules to import unmodified:
  _methods.dinov2.{dinov2_loss,dinov2_head,utils,scheduler}, _models.dinov2_vit.dinov2_vit_src.*, _torch_helpers.
Only the fixture generators under tools/ use this; the tests read what they wrote under tests/golden/.
"""
from __future__ import annotations

import os
import sys
import types
from pathlib import Path

REF_SRC = Path(os.environ.get("LIGHTLY_TRAIN_SRC", "")) / "lightly_train"


def available() -> bool:
    try:
        return "LIGHTLY_TRAIN_SRC" in os.environ and REF_SRC.is_dir()
    except OSError:
        return False


def install() -> None:
    if "lightly_train" in sys.modules:
        return
    if not available():
        raise RuntimeError("set LIGHTLY_TRAIN_SRC to the src directory of a lightly-train checkout")
    os.environ["XFORMERS_DISABLED"] = "1"
    pkg = types.ModuleType("lightly_train")
    pkg.__path__ = [str(REF_SRC)]  # namespace-style: skips lightly_train/__init__.py
    sys.modules["lightly_train"] = pkg
    if "lightning_utilities" not in sys.modules:
        lu = types.ModuleType("lightning_utilities")
        core = types.ModuleType("lightning_utilities.core")
        imports = types.ModuleType("lightning_utilities.core.imports")

        class RequirementCache:  # minimal stand-in: every optional requirement is "not installed"
            def __init__(self, *a, **k):
                pass

            def __bool__(self):
                return False

        imports.RequirementCache = RequirementCache
        lu.core = core
        core.imports = imports
        sys.modules.update({"lightning_utilities": lu, "lightning_utilities.core": core,
                            "lightning_utilities.core.imports": imports})


def modules():
    """Return the reference modules the oracle is pinned against."""
    install()
    from lightly_train._methods.dinov2 import dinov2_head, dinov2_loss, scheduler, utils  # type: ignore
    from lightly_train._models.dinov2_vit.dinov2_vit_src.models import vision_transformer  # type: ignore
    from lightly_train import _torch_helpers  # type: ignore

    return types.SimpleNamespace(head=dinov2_head, loss=dinov2_loss, scheduler=scheduler, utils=utils,
                                 vit=vision_transformer, torch_helpers=_torch_helpers)
