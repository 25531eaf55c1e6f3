"""Build libplaid_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libplaid_b200.so")
SOURCES = ["engine.cu", "loader.cpp", "builder.cpp"]
DEPS = SOURCES + sorted(f for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))) + \
    [os.path.join("..", "..", "include", "plaid_b200.h")]
NVCC_FLAGS = [
    "-shared", "-std=c++17", "-O3", "-lineinfo",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-Xcompiler", "-fPIC,-fvisibility=hidden",
]


def cuda_tool(name: str) -> str:
    """A CUDA toolkit program: from PATH, else from $CUDA_HOME/bin (default /usr/local/cuda), where the toolkit
    installs it even when a user's PATH does not name that directory."""
    found = shutil.which(name)
    if found:
        return found
    home = os.environ.get("CUDA_HOME") or os.environ.get("CUDA_PATH") or "/usr/local/cuda"
    path = os.path.join(home, "bin", name)
    if not os.access(path, os.X_OK):
        raise RuntimeError(f"{name} is neither on PATH nor in {os.path.dirname(path)}; set CUDA_HOME")
    return path


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC") or cuda_tool("nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          [os.path.join(CSRC, s) for s in SOURCES] + ["-o", LIB]
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout)
    if verbose:
        print(r.stdout)
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
