"""Recipe for ``oracle/_ref``: a runnable copy of the reference's own Python package.

TEST / BENCH INFRASTRUCTURE ONLY.  ``python oracle/make_ref.py <reference checkout>`` copies
``<reference checkout>/src/aggforce`` UNMODIFIED into ``oracle/_ref/aggforce``.  ``oracle/_ref/``
is git-ignored (reference sources never enter the history); where it exists, ``bench.py --impl
reference`` and ``bench.py``'s ``cpu_baseline`` leg time the reference's own
``guess_pairwise_constraints`` / ``project_forces`` on the host cores, and where it does not they
time the numpy port in ``oracle/``.

The reference imports ``qpsolvers`` (absent here, unpinned in its ``setup.cfg``); ``load()`` installs
``oracle/qpsolvers_shim.py`` -- the exact equality-QP solve -- under that name before importing it.
Its JAX-guarded modules drop out on import (``try/except ImportError`` in the reference's own
``__init__`` files); the timed path is numpy only.
"""
from __future__ import annotations

import shutil
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
DEST = HERE / "_ref"


def make(reference: str | Path) -> Path:
    """Copy the package ``<reference>/src/aggforce`` of a reference checkout; returns the destination."""
    src = Path(reference) / "src" / "aggforce"
    if not src.is_dir():
        raise FileNotFoundError(f"{src} is not a directory: pass the root of an aggforce checkout")
    if DEST.exists():
        shutil.rmtree(DEST)
    DEST.mkdir(parents=True)
    shutil.copytree(src, DEST / "aggforce", ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    (DEST / "README").write_text(
        "Unmodified copy of the reference's src/aggforce made by oracle/make_ref.py; git-ignored, not product.\n")
    return DEST


def available() -> bool:
    return (DEST / "aggforce" / "__init__.py").exists()


def load():
    """Import the reference package from ``oracle/_ref`` (behind the qpsolvers shim); ``None`` if absent."""
    if not available():
        return None
    if "qpsolvers" not in sys.modules:
        from . import qpsolvers_shim

        sys.modules["qpsolvers"] = qpsolvers_shim
    if str(DEST) not in sys.path:
        sys.path.insert(0, str(DEST))
    import aggforce  # noqa: PLC0415  (the reference)

    assert str(DEST) in str(Path(aggforce.__file__).resolve()), aggforce.__file__
    return aggforce


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python oracle/make_ref.py <reference checkout>")
    print(make(sys.argv[1]))
