"""Import the *unmodified* reference librosa from /root/reference in this container.

Build-container-only helper (the GPU box has no /root/reference). It is used by
``tools/make_golden.py`` to generate the committed fixtures under ``tests/golden/``, against which
the tests pin the ``oracle/`` restatement; no test imports the reference itself.

librosa imports four modules at import time that are missing from the image and never called on
the stft / istft / melspectrogram / mfcc path (``lazy_loader``, ``soundfile``, ``soxr``, ``pooch``);
they are replaced by in-memory stubs. Nothing from the reference is copied into this repository.
"""
from __future__ import annotations

import ast
import importlib
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("B2L_REFERENCE_ROOT", "/root/reference")


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "librosa"))


def _stub_lazy_loader() -> types.ModuleType:
    mod = types.ModuleType("lazy_loader")

    def attach_stub(package_name: str, filename: str):
        """Resolve names listed in the sibling ``.pyi`` on first attribute access."""
        stub = os.path.splitext(filename)[0] + ".pyi"
        with open(stub, "r", encoding="utf-8") as fh:
            tree = ast.parse(fh.read())
        attr_to_mod: dict[str, str] = {}
        submodules: set[str] = set()
        for node in tree.body:
            if isinstance(node, ast.ImportFrom) and node.level == 1:
                if node.module is None:
                    for alias in node.names:
                        submodules.add(alias.asname or alias.name)
                else:
                    for alias in node.names:
                        attr_to_mod[alias.asname or alias.name] = node.module
        names = sorted(submodules | set(attr_to_mod))

        def __getattr__(name: str):
            if name in submodules:
                return importlib.import_module(f"{package_name}.{name}")
            if name in attr_to_mod:
                sub = importlib.import_module(f"{package_name}.{attr_to_mod[name]}")
                return getattr(sub, name)
            raise AttributeError(f"No {package_name} attribute {name}")

        def __dir__():
            return names

        return __getattr__, __dir__, names

    def load(name: str, *args, **kwargs):
        return types.ModuleType(name)

    mod.attach_stub = attach_stub
    mod.load = load
    return mod


def _stub_pooch() -> types.ModuleType:
    mod = types.ModuleType("pooch")

    class _Registry:
        registry: dict = {}

        def load_registry(self, *a, **k):
            return None

        def fetch(self, *a, **k):
            raise RuntimeError("pooch stub: no network / no example data")

    mod.os_cache = lambda name: os.path.join("/tmp", name)
    mod.create = lambda *a, **k: _Registry()
    return mod


def load_reference():
    """Return the reference ``librosa`` module (raises if /root/reference is absent)."""
    if not available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    if "librosa" in sys.modules and getattr(sys.modules["librosa"], "__b2l_reference__", False):
        return sys.modules["librosa"]
    os.environ.setdefault("NUMBA_CACHE_DIR", "/tmp/b2l_numba_cache")
    sys.modules.setdefault("lazy_loader", _stub_lazy_loader())
    sys.modules.setdefault("pooch", _stub_pooch())
    for name in ("soundfile", "soxr"):
        sys.modules.setdefault(name, types.ModuleType(name))
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import librosa  # noqa: E402  (the reference, from /root/reference)

    librosa.__b2l_reference__ = True
    return librosa


if __name__ == "__main__":
    import numpy as np

    ref = load_reference()
    y = np.random.default_rng(0).standard_normal(22050).astype(np.float32)
    D = ref.stft(y)
    M = ref.feature.melspectrogram(y=y, sr=22050)
    C = ref.feature.mfcc(y=y, sr=22050)
    yr = ref.istft(D, length=len(y))
    print("reference", ref.__version__, D.shape, D.dtype, M.shape, C.shape, float(np.abs(y - yr).max()))
