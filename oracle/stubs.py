"""ORACLE / TEST INFRASTRUCTURE — not part of the shipped product.

sys.modules stubs for the packages the reference imports at module scope but never touches on the
reward-labeling path (SURVEY.md §8c): gcsfs, ml_collections(+config_dict, config_flags), flax,
jax(+numpy), kornia.augmentation.ColorJitter (train-only augmentation, identity here), wandb.
Also puts oracle/shims (clip, h5py) ahead on sys.path unless the real packages are importable.
"""
from __future__ import annotations

import importlib
import importlib.util
import os
import sys
import types
from pathlib import Path

HERE = Path(__file__).resolve().parent
REFERENCE = Path("/root/reference")


class _Auto(types.ModuleType):
    """Module whose every attribute is another auto-module / a do-nothing callable class."""

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        val = type(name, (), {"__init__": lambda self, *a, **k: None, "__call__": lambda self, *a, **k: None})
        setattr(self, name, val)
        return val


def _stub(name: str):
    if name in sys.modules:
        return sys.modules[name]
    try:
        if importlib.util.find_spec(name) is not None:
            return None
    except (ImportError, ValueError):
        pass
    m = _Auto(name)
    m.__path__ = []  # behave like a package so `import a.b` resolves through sys.modules
    sys.modules[name] = m
    parent, _, child = name.rpartition(".")
    if parent and parent in sys.modules:
        setattr(sys.modules[parent], child, m)
    return m


def install(use_shims: bool = True):
    for name in ("gcsfs", "ml_collections", "ml_collections.config_dict", "ml_collections.config_flags", "flax",
                 "jax", "jax.numpy", "wandb", "kornia", "kornia.augmentation"):
        _stub(name)
    if "kornia.augmentation" in sys.modules and isinstance(sys.modules["kornia.augmentation"], _Auto):
        import torch

        class ColorJitter(torch.nn.Module):  # identity: only used with train=True (clip_multiscale_adapter.py:128)
            def __init__(self, *a, **k):
                super().__init__()

            def forward(self, x):
                return x

        sys.modules["kornia.augmentation"].ColorJitter = ColorJitter
    if use_shims:
        shim = str(HERE / "shims")
        if shim not in sys.path:
            sys.path.insert(0, shim)


def reference_available() -> bool:
    return os.path.exists(REFERENCE / "arp_dt" / "label_reward.py")     # False, not an error, where it is unreadable


def import_reference():
    """Import the reference's own modules (only possible where /root/reference is mounted)."""
    install()
    if str(REFERENCE) not in sys.path:
        sys.path.insert(0, str(REFERENCE))
    lr = importlib.import_module("arp_dt.label_reward")
    return lr
