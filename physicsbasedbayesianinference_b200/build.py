"""In-tree build of the CUDA library (``_ehmc.so``) for sm_100a with nvcc.

    python -m physicsbasedbayesianinference_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU
box with the repository snapshot.
"""
from __future__ import annotations

import glob
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "_ehmc.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC,-fvisibility=hidden", "-cudart", "static",
]


def cuda_tool(name):
    """Path of a CUDA toolkit program: on PATH, else under $CUDA_HOME (or $CUDA_PATH, or /usr/local/cuda)/bin,
    which is where the toolkit lives when a login shell does not put it on PATH."""
    found = shutil.which(name)
    if found:
        return found
    home = os.environ.get("CUDA_HOME") or os.environ.get("CUDA_PATH") or "/usr/local/cuda"
    path = os.path.join(home, "bin", name)
    if not os.path.isfile(path):
        raise FileNotFoundError(f"{name} is neither on PATH nor in {os.path.dirname(path)}: set CUDA_HOME")
    return path


def _sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def _deps(path, seen=None):
    """The file plus every header it includes with quotes, recursively."""
    import re

    seen = set() if seen is None else seen
    if path in seen or not os.path.isfile(path):
        return seen
    seen.add(path)
    with open(path) as f:
        for inc in re.findall(r'^\s*#include\s+"([^"]+)"', f.read(), flags=re.M):
            _deps(os.path.normpath(os.path.join(os.path.dirname(path), inc)), seen)
    return seen


def _newer(target, sources):
    if not os.path.isfile(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def build_library(force=False, verbose=False):
    """Compile the .cu files under csrc/ that changed (parallel per file) and link one shared library."""
    nvcc = os.environ.get("NVCC") or cuda_tool("nvcc")
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    objs = []
    for src in _sources():
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        if not force and not _newer(obj, _deps(src) | {os.path.abspath(__file__)}):
            continue
        cmd = [nvcc, *NVCC_FLAGS, "-I", INCLUDE, "-c", src, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}")
    if procs or force or _newer(OUT, objs):
        cmd = [nvcc, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a", "-o", OUT, *objs]
        subprocess.run(cmd, check=True)
    return OUT


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
