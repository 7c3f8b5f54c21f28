"""Build ``oracle/_ref``: the unmodified pulser-core package of an upstream Pulser source checkout.

pulser-core (Sequence, sampler, HamiltonianData, NoiseModel) is the input layer of the facade and of the tests that
drive it with real ``pulser.Sequence`` objects. It is pure Python, so building it is a copy of its package tree, laid
out as in the checkout (``_ref/VERSION.txt`` beside ``_ref/pulser-core/pulser/``) because ``pulser/_version.py``
reads the version file two directories above itself. ``oracle/_ref`` is git-ignored; once built it travels with the
working tree, so machines without the checkout import pulser from it (``pulser_b200/_compat.py``).

The checkout is looked up at ``$PULSER_B200_REFERENCE_SRC``, by default ``/root/reference``. Where it is not readable
and ``oracle/_ref`` was not built before, nothing is built and the pulser-driven tests skip.
"""
from __future__ import annotations

import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, "_ref")
CORE = os.path.join(DEST, "pulser-core")
DEFAULT_SRC = "/root/reference"


def built() -> bool:
    return os.path.isfile(os.path.join(CORE, "pulser", "__init__.py")) and os.path.isfile(os.path.join(DEST, "VERSION.txt"))


def source() -> str | None:
    root = os.environ.get("PULSER_B200_REFERENCE_SRC") or DEFAULT_SRC
    ok = os.path.isfile(os.path.join(root, "VERSION.txt")) and os.path.isfile(
        os.path.join(root, "pulser-core", "pulser", "__init__.py"))
    return root if ok else None


def _copy_tree(src: str, dst: str) -> None:
    """File contents only: the checkout may be read-only, the copy stays writable (and removable) by its owner."""
    for dirpath, dirnames, filenames in os.walk(src):
        dirnames[:] = [d for d in dirnames if d != "__pycache__"]
        out = os.path.join(dst, os.path.relpath(dirpath, src))
        os.makedirs(out, exist_ok=True)
        for f in filenames:
            if not f.endswith(".pyc"):
                shutil.copyfile(os.path.join(dirpath, f), os.path.join(out, f))


def build() -> bool:
    """Make ``oracle/_ref`` if it is missing and the checkout is readable. Returns whether it holds pulser-core."""
    if built():
        return True
    src = source()
    if src is None:
        return False
    partial = os.path.join(DEST, "pulser-core.partial")
    shutil.rmtree(partial, ignore_errors=True)
    _copy_tree(os.path.join(src, "pulser-core", "pulser"), os.path.join(partial, "pulser"))
    shutil.copyfile(os.path.join(src, "VERSION.txt"), os.path.join(DEST, "VERSION.txt"))
    shutil.rmtree(CORE, ignore_errors=True)
    os.rename(partial, CORE)
    return True


if __name__ == "__main__":
    ok = build()
    print(CORE if ok else "pulser-core checkout not found: set PULSER_B200_REFERENCE_SRC", file=sys.stdout if ok else sys.stderr)
    sys.exit(0 if ok else 1)
