#!/usr/bin/env python
"""Copy the UNMODIFIED reference into baseline/_ref/ (git-ignored).

    MAZE_REFERENCE_ROOT=<checkout of the reference> python tools/install_reference.py

The reference has no setup.py / pyproject.toml, so there is nothing to pip-install (DESIGN.md section 5); a plain
copy of its Python tree is the install.  baseline/_ref is bench infrastructure: where it is present,
`bench.py --impl reference` times the reference's own SimpleMazeEnv instead of the oracle's port of it.  Nothing under
maze-solving-agent-gymnasium_b200/ reads it, and none of it is committed.
"""
from __future__ import annotations

import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.environ.get("MAZE_REFERENCE_ROOT", "/root/reference")
DST = os.path.join(ROOT, "baseline", "_ref")
TREES = ("agents", "lib", "gymnasium_env", "training_examples")


def install(verbose: bool = True) -> bool:
    if not os.path.isdir(os.path.join(SRC, "gymnasium_env")):
        if verbose:
            print(f"reference not found at {SRC}: leaving {DST} as it is")
        return False
    os.makedirs(DST, exist_ok=True)
    for t in TREES:
        dst = os.path.join(DST, t)
        if os.path.isdir(dst):
            shutil.rmtree(dst)
        shutil.copytree(os.path.join(SRC, t), dst, ignore=shutil.ignore_patterns("__pycache__", "*.pyc", "weights", "logs"))
    for f in os.listdir(SRC):
        if f.endswith(".py") or f == "README.md":
            shutil.copy2(os.path.join(SRC, f), os.path.join(DST, f))
    if verbose:
        print(f"copied {', '.join(TREES)} from {SRC} to {DST}")
    return True


if __name__ == "__main__":
    sys.exit(0 if install() else 1)
