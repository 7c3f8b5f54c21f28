"""Locate and import the real ``pulser`` (pulser-core) package, headless.

pulser-core is reused unmodified as the *input layer* (Sequence, sampler,
HamiltonianData, NoiseModel): everything upstream of
``pulser_simulation.hamiltonian.Hamiltonian.__init__`` (SURVEY.md section 0.3).
Its only hard non-numeric dependency is matplotlib (drawing only,
``pulser-core/pulser/waveforms.py:28``), which is absent from this image, so a
meta-path finder serves empty stand-in modules for ``matplotlib.*``.

pulser is OPTIONAL: the CUDA path, the C-ABI and the plain-array
``HamiltonianSpec`` entry point work without it.
"""
from __future__ import annotations

import importlib.abc
import importlib.machinery
import importlib.util
import os
import sys
import types

# copy of the unmodified pulser-core that build() makes with oracle/ref_build.py (git-ignored, DESIGN.md section 5)
_BUILT_CORE = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "pulser-core")


class _Anything:
    """Placeholder for any attribute of a stubbed drawing module."""

    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        return _Anything()

    def __getattr__(self, name):
        if name.startswith("__") and name.endswith("__"):
            raise AttributeError(name)
        return _Anything()

    def __iter__(self):
        return iter(())

    def __mro_entries__(self, bases):
        return (object,)


class _StubModule(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__") and name.endswith("__"):
            raise AttributeError(name)
        return _Anything


class _StubLoader(importlib.abc.Loader):
    def create_module(self, spec):
        mod = _StubModule(spec.name)
        mod.__path__ = []  # behave as a package
        return mod

    def exec_module(self, module):
        pass


class _DrawingStubFinder(importlib.abc.MetaPathFinder):
    _TOPS = ("matplotlib", "mpl_toolkits")

    def find_spec(self, fullname, path=None, target=None):
        if fullname.split(".")[0] in self._TOPS:
            return importlib.machinery.ModuleSpec(
                fullname, _StubLoader(), is_package=True
            )
        return None


def _have(modname: str) -> bool:
    try:
        return importlib.util.find_spec(modname) is not None
    except (ImportError, ValueError):
        return False


def ensure_pulser() -> bool:
    """Make ``import pulser`` work if a copy is reachable. Returns success."""
    if "pulser" in sys.modules:
        return True
    if not _have("matplotlib"):
        if not any(isinstance(f, _DrawingStubFinder) for f in sys.meta_path):
            sys.meta_path.append(_DrawingStubFinder())
    if not _have("pulser"):
        for root in (os.environ.get("PULSER_B200_PULSER_PATH"), _BUILT_CORE):
            if root and os.path.isdir(os.path.join(root, "pulser")):
                sys.path.insert(0, root)
                break
        else:
            return False
    try:
        import pulser  # noqa: F401
    except Exception:  # pragma: no cover - environment dependent
        return False
    return True


HAVE_PULSER = ensure_pulser()
