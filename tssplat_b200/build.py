"""In-tree build of ``libtssplat_b200.so`` (the C-ABI library) with nvcc for sm_100a.

``python -m tssplat_b200.build`` or ``__graft_entry__.build()``.  The .so stays in-tree
(git-ignored) so it travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, "libtssplat_b200.so")
SOURCES = ["tsb_plan.cpp", "tsb_kernels.cu", "tsb_capi.cu", "tsb_surface.cu", "tsb_setup.cu", "tsb_train.cu"]
HEADERS = ["tsb_plan.h", "tsb_kernels.cuh", os.path.join("..", "..", "include", "tssplat_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC,-O2,-Wall",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA library cannot be built (no CPU fallback exists)")


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False, extra_flags=()) -> str:
    if not force and not needs_build():
        return LIB_PATH
    cmd = [_nvcc(), *NVCC_FLAGS, *extra_flags, "-shared", "-o", LIB_PATH,
           *[os.path.join(CSRC, s) for s in SOURCES]]
    if verbose:
        print(" ".join(cmd), file=sys.stderr)
    env = dict(os.environ)
    env.pop("CC", None)      # this image's $CC wrapper lacks the OpenMP spec; nvcc needs none of it
    env.pop("CXX", None)
    res = subprocess.run(cmd, capture_output=True, text=True, env=env)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose and (res.stdout or res.stderr):
        print(res.stdout + res.stderr, file=sys.stderr)
    return LIB_PATH


if __name__ == "__main__":
    flags = ["-Xptxas", "-v"] if "-v" in sys.argv else []
    print(build_library(force=True, verbose=True, extra_flags=flags))
