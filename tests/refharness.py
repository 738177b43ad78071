"""Harness (test infrastructure only) for running the reference's OWN Python files unchanged.

The reference (the original LiDOG sources) is not part of this repository: put a checkout of it at oracle/_ref/
(git-ignored) to run them.  These helpers are used by CPU tests that skip when it is absent, and by
tests/golden/make_*_golden.py, which commit what the reference computes as fixtures.

The reference's files import `MinkowskiEngine`, `pytorch_lightning` and `torchmetrics` (SURVEY.md Appendix D).  The
first is bound to the module under test (the CPU oracle shim or the CUDA product), the other two to the minimal
stand-ins below -- exactly what `PLTTrainer2D` touches (`trainer_lighting_2d.py:4,6,75`, `:141-360`).  Nothing of the
reference is copied: its files are imported from where they lie."""
from __future__ import annotations

import contextlib
import importlib
import importlib.util
import os
import sys
import types

import torch

REF = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REF, "utils", "models"))


class _LightningModule(torch.nn.Module):
    """pl.core.LightningModule as far as PLTTrainer2D uses it."""

    def __init__(self):
        super().__init__()
        self.logged = {}
        self.global_step = 0
        self.current_epoch = 0
        self.trainer = types.SimpleNamespace(optimizers=[])

    def log(self, name, value, **kw):
        self.logged[name] = float(value)

    def save_hyperparameters(self, *a, **kw):
        pass

    @property
    def device(self):
        p = next(self.parameters(), None)
        return p.device if p is not None else torch.device("cpu")


class _JaccardIndex:
    """torchmetrics.JaccardIndex(num_classes, ignore_index, average='none'): per-class IoU of two label vectors."""

    def __init__(self, num_classes, ignore_index=None, average="none", **kw):
        self.num_classes, self.ignore_index = num_classes, ignore_index

    def __call__(self, preds, target):
        preds, target = preds.reshape(-1), target.reshape(-1)
        if self.ignore_index is not None:
            keep = target != self.ignore_index
            preds, target = preds[keep], target[keep]
        out = torch.zeros(self.num_classes, device=preds.device)
        for c in range(self.num_classes):
            inter = ((preds == c) & (target == c)).sum()
            union = ((preds == c) | (target == c)).sum()
            out[c] = inter.float() / union.clamp_min(1).float()
        return out


def _stub_modules():
    pl = types.ModuleType("pytorch_lightning")
    pl.core = types.ModuleType("pytorch_lightning.core")
    pl.core.LightningModule = _LightningModule
    pl.LightningModule = _LightningModule
    tm = types.ModuleType("torchmetrics")
    tm.JaccardIndex = _JaccardIndex
    return {"pytorch_lightning": pl, "pytorch_lightning.core": pl.core, "torchmetrics": tm}


@contextlib.contextmanager
def reference(me_module):
    """sys.path / sys.modules set up so that the reference's files import `me_module` as MinkowskiEngine."""
    saved = {k: sys.modules.get(k) for k in ("MinkowskiEngine", "MinkowskiEngine.modules",
                                             "MinkowskiEngine.modules.resnet_block", "MinkowskiEngine.utils",
                                             "pytorch_lightning", "pytorch_lightning.core", "torchmetrics")}
    for k in [k for k in sys.modules if k == "utils" or k.startswith("utils.")]:
        saved[k] = sys.modules.pop(k)
    sys.modules["MinkowskiEngine"] = me_module
    for sub in ("modules", "utils"):
        if hasattr(me_module, sub):
            sys.modules["MinkowskiEngine." + sub] = getattr(me_module, sub)
    if hasattr(me_module, "modules") and hasattr(me_module.modules, "resnet_block"):
        sys.modules["MinkowskiEngine.modules.resnet_block"] = me_module.modules.resnet_block
    sys.modules.update(_stub_modules())
    sys.path.insert(0, REF)
    try:
        yield
    finally:
        sys.path.remove(REF)
        for k in [k for k in sys.modules if k == "utils" or k.startswith("utils.") or k.startswith("_lidog_ref_")]:
            del sys.modules[k]
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def load_file(relpath: str, name: str):
    """Import ONE reference file by path (its package __init__ would pull open3d / wandb / the nuScenes devkit)."""
    spec = importlib.util.spec_from_file_location("_lidog_ref_" + name, os.path.join(REF, relpath))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[spec.name] = mod
    spec.loader.exec_module(mod)
    return mod


class FakeDataset:
    """What PLTTrainer2D reads from its datasets (`ignore_label`, `class2names`)."""
    ignore_label = -1

    def __init__(self, num_classes=7):
        import numpy as np
        self.class2names = np.array(["ignore"] + [f"class{i}" for i in range(num_classes)])
