"""Recipe for oracle/_ref: the UNMODIFIED reference package, so that `bench.py --impl reference` can time the
reference's own `ScorerPress.compress` (kvpress/presses/scorer_press.py:76-102) on the GPU box's host cores.

TEST / MEASUREMENT INFRASTRUCTURE ONLY — nothing under kvpress_b200/ may import this.

The reference is pure Python (no build step): the recipe copies `/root/reference/kvpress` as it is into
`oracle/_ref/kvpress` and adds a one-line `fire` stub module (the reference imports `fire` at package import for
an unrelated CLI, SURVEY §8c; `fire` is not installed in this image). `oracle/_ref/` is git-ignored (reference
sources never enter the history) but not gpurun-ignored, so it travels to the GPU box with the snapshot.
Run in the build container, where /root/reference exists:  python oracle/build_ref.py
"""
from __future__ import annotations

import os
import shutil
import sys
from pathlib import Path

REFERENCE = Path("/root/reference")
DEST = Path(__file__).resolve().parent / "_ref"


def build_ref(force: bool = False) -> Path | None:
    """Returns oracle/_ref (built if needed), or None when there is no reference checkout to take it from."""
    marker = DEST / "kvpress" / "__init__.py"
    if marker.exists() and not force:
        return DEST
    if not os.path.isfile(REFERENCE / "kvpress" / "__init__.py"):     # absent, or not readable by this user
        return DEST if marker.exists() else None
    if DEST.exists():
        shutil.rmtree(DEST)
    DEST.mkdir(parents=True)
    shutil.copytree(REFERENCE / "kvpress", DEST / "kvpress", ignore=shutil.ignore_patterns("__pycache__"))
    (DEST / "fire.py").write_text('"""stub: the reference imports `fire` for a CLI entry point that is never used here"""\n')
    (DEST / "README").write_text("unmodified copy of /root/reference/kvpress made by oracle/build_ref.py; git-ignored\n")
    return DEST


def import_ref():
    """The reference package from oracle/_ref (None if it was never built). Importing it wraps transformers'
    attention functions (kvpress/__init__.py:52) exactly like the reference does in its own process."""
    if not (DEST / "kvpress" / "__init__.py").exists():
        return None
    if str(DEST) not in sys.path:
        sys.path.insert(0, str(DEST))
    import kvpress  # noqa: the reference

    return kvpress


if __name__ == "__main__":
    print(build_ref(force="--force" in sys.argv))
