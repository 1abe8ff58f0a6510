"""Build libmaze_b200.so (sm_100a only) in-tree with nvcc."""
from __future__ import annotations

import os
import shutil
import subprocess

PKG_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REPO_ROOT = os.path.dirname(PKG_ROOT)
CSRC = os.path.join(PKG_ROOT, "csrc")
# MAZE_B200_LIB: load another build of the same ABI (e.g. one written with build(out=...), to compare two
# builds); default in-tree .so
LIB_PATH = os.environ.get("MAZE_B200_LIB") or os.path.join(PKG_ROOT, "libmaze_b200.so")
INCLUDE = os.path.join(REPO_ROOT, "include")


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "maze_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, out=None) -> str:
    if out is None and not force and not needs_build():
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
           "--compiler-options", "-fPIC", "-shared", "-I", INCLUDE, "-I", CSRC, "-o", out or LIB_PATH]
    cmd += sources()
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return out or LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
