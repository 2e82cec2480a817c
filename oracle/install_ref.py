"""TEST INFRASTRUCTURE.  Copies the unmodified original project (facebookresearch/SlowFast) into ``oracle/_ref`` (git-ignored),
where ``oracle/refshim.py`` finds it for the tests and baselines that run the original code itself (driver tests,
registry integration, bench.py's CPU and ATen-GPU baselines).

    python oracle/install_ref.py          # also run by build()

The source checkout is ``$SLOWFAST_REFERENCE_SRC`` (default ``/root/reference``, as baseline/install_ref.sh).  Its
``slowfast`` package is pure Python, so the install is a verbatim copy of it, as ``pip install --no-deps`` would make,
plus the files of the checkout the tests use next to it: ``tools/`` (train_net.py, test_net.py), ``configs/`` and
``ava_evaluation/``.  Nothing is edited.  Without a readable checkout nothing is done and an existing install is kept.
"""
from __future__ import annotations

import os
import shutil
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEST = os.path.join(ROOT, "oracle", "_ref")
PARTS = ("slowfast", "tools", "configs", "ava_evaluation")


def source() -> str:
    return os.environ.get("SLOWFAST_REFERENCE_SRC", "/root/reference")


def install() -> str | None:
    """Copy the checkout into oracle/_ref; returns the install path, or None when there is no readable checkout."""
    src = source()
    if not all(os.access(os.path.join(src, p), os.R_OK | os.X_OK) for p in PARTS):
        return None
    tmp = tempfile.mkdtemp(prefix="_ref.", dir=os.path.dirname(DEST))
    try:
        for p in PARTS:
            shutil.copytree(os.path.join(src, p), os.path.join(tmp, p),
                            ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
        os.chmod(tmp, 0o755)
        if os.path.isdir(DEST):
            shutil.rmtree(DEST)
        os.rename(tmp, DEST)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return DEST


if __name__ == "__main__":
    print(install() or f"no readable checkout at {source()}: nothing installed")
