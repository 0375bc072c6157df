"""TEST INFRASTRUCTURE ONLY -- import the real reference (georghess/neurad-studio) in THIS container.

The reference lives read-only at /root/reference and is pure Python on top of torch, but it hard-imports
third-party packages that are absent here (viser, nerfacc, tinycudann, gsplat, torchmetrics ...).  SURVEY.md
section 8(c) lists the modules that have to be stubbed in ``sys.modules`` before
``nerfstudio.models.neurad`` imports cleanly.  This module installs those stubs and puts /root/reference on
``sys.path``.

It is used by ``oracle/make_golden.py`` (fixture generation) and by the CPU-side oracle self-checks; it never
runs on the GPU box (``/root/reference`` does not exist there) and nothing under ``neurad-studio_b200/`` may
import it.
"""
from __future__ import annotations

import importlib.machinery
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("NEURAD_REFERENCE_ROOT", "/root/reference")

_STUBS = [
    "viser", "viser.transforms", "viser.theme", "viser.infra",
    "nerfacc",
    "matplotlib", "matplotlib.pyplot", "matplotlib.cm",
    "torchmetrics", "torchmetrics.functional", "torchmetrics.image", "torchmetrics.image.lpip",
    "pyquaternion", "h5py", "mediapy", "plotly", "plotly.graph_objects", "open3d", "wandb", "comet_ml",
    "pytorch_msssim", "gsplat", "timm", "torch.utils.tensorboard", "tinycudann",
]


# further absent third-party packages that only the FULL method registry (nerfstudio.configs.method_configs: every
# dataparser and model of the reference) pulls in; needed by oracle/make_golden_reference_recipe.py
_STUBS_FULL = [
    "av2", "av2.utils", "av2.utils.io", "av2.datasets", "av2.datasets.sensor", "av2.datasets.sensor.av2_sensor_dataloader",
    "av2.datasets.sensor.constants", "av2.geometry", "av2.geometry.geometry", "av2.structures", "av2.structures.sweep",
    "nuscenes", "nuscenes.nuscenes", "pandaset", "zod", "zod.constants", "zod.data_classes", "zod.data_classes.box",
    "zod.data_classes.sensor", "pathos", "pathos.helpers", "gsplat.strategy", "gsplat.strategy.ops", "splines",
    "splines.quaternion", "imageio", "imageio.v3", "torchmetrics.image.fid",
]


class _Anything:
    """Attribute sink: any attribute / call / subscript returns another sink (enough for import-time use)."""

    def __init__(self, name="stub"):
        self.__name__ = name

    def __getattr__(self, item):
        if item.startswith("__") and item.endswith("__"):
            raise AttributeError(item)
        return _Anything(f"{self.__name__}.{item}")

    def __call__(self, *a, **k):
        return _Anything(self.__name__ + "()")

    def __getitem__(self, item):
        return _Anything(self.__name__ + "[]")

    def __mro_entries__(self, bases):
        return (object,)


class _StubModule(types.ModuleType):
    def __getattr__(self, item):
        if item.startswith("__") and item.endswith("__"):
            raise AttributeError(item)
        return _Anything(f"{self.__name__}.{item}")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "nerfstudio"))


def install(full: bool = False) -> None:
    """Install the stubs and make ``import nerfstudio`` resolve to the reference tree.  ``full``: also the packages the
    complete method registry imports (``nerfstudio.configs.method_configs`` / ``nerfstudio.plugins.registry``)."""
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT} (only present in the build container)")
    for name in _STUBS + (_STUBS_FULL if full else []):
        if name in sys.modules:
            continue
        if name == "tinycudann":
            # must stay un-importable so that utils/external.py sets TCNN_EXISTS = False
            continue
        mod = _StubModule(name)
        mod.__spec__ = importlib.machinery.ModuleSpec(name, loader=None)
        mod.__path__ = []  # behave like a package so that submodule imports work
        sys.modules[name] = mod
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
