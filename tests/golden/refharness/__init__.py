"""TEST INFRASTRUCTURE: import the read-only MAC-VO reference tree (MACVO_REFERENCE_ROOT).

Used only by the fixture generators `tests/golden/make_golden*.py`; the tests read the fixtures they
write and never need the tree. Nothing in the product imports this.

* `yacs` is absent -> tiny `CfgNode` stand-in (`refharness/yacs`).
* `pypose` is absent -> functional restatement (`oracle/pypose_shim`).
* `matplotlib`, `evo`, `rerun`, `flow_vis`, `mpl_toolkits`, `cv2` (if absent) -> permissive auto-stubs:
  only needed so that `import Module` / `import DataLoader` succeed; never executed on the hot path.
"""
from __future__ import annotations

import importlib.abc
import importlib.machinery
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("MACVO_REFERENCE_ROOT", "/root/reference")
_HERE = os.path.dirname(os.path.abspath(__file__))
_REPO = os.path.dirname(os.path.dirname(os.path.dirname(_HERE)))
_AUTO_STUB_ROOTS = ("matplotlib", "evo", "flow_vis", "mpl_toolkits", "cv2", "wandb", "kornia")   # rerun is optional in MAC-VO (ImportError -> None)


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "Module"))


class _StubMeta(type):
    def __getattr__(cls, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _make_stub(name)

    def __or__(cls, other):
        return cls

    def __ror__(cls, other):
        return cls


def _make_stub(name: str):
    return _StubMeta(name, (), {"__init__": lambda self, *a, **k: None,
                                "__call__": lambda self, *a, **k: self,
                                "__getattr__": lambda self, n: _make_stub(n)(),
                                "__iter__": lambda self: iter(()),
                                "__getitem__": lambda self, k: self,
                                "__enter__": lambda self: self,
                                "__exit__": lambda self, *a: False})


class _StubModule(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _make_stub(name)


class _AutoStubFinder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    def find_spec(self, fullname, path=None, target=None):
        if fullname.split(".")[0] in _AUTO_STUB_ROOTS:
            return importlib.machinery.ModuleSpec(fullname, self, is_package=True)
        return None

    def create_module(self, spec):
        m = _StubModule(spec.name)
        m.__path__ = []
        return m

    def exec_module(self, module):
        pass


_installed = False


def install(full: bool = True) -> None:
    """Make `import Module, DataLoader, Utility, Odometry` (full) or the network sub-packages work."""
    global _installed, _AUTO_STUB_ROOTS
    if _installed:
        return
    if not available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    os.environ.setdefault("TORCHDYNAMO_DISABLE", "1")
    # really-installed packages win; only stub what is missing
    missing = []
    for root in _AUTO_STUB_ROOTS:
        try:
            __import__(root)
        except Exception:
            missing.append(root)
    _AUTO_STUB_ROOTS = tuple(missing)
    sys.meta_path.append(_AutoStubFinder())
    try:
        import yacs  # noqa: F401
    except Exception:
        sys.path.insert(0, _HERE)  # exposes refharness/yacs as top-level `yacs`
    try:
        import pypose  # noqa: F401
    except Exception:
        sys.path.insert(0, os.path.join(_REPO, "oracle", "pypose_shim"))
    if REFERENCE_ROOT not in sys.path:
        sys.path.append(REFERENCE_ROOT)
    _installed = True
