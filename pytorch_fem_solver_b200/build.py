"""In-tree build of the CUDA library behind include/tfem_b200.h (sm_100a only).

`python -m pytorch_fem_solver_b200.build` or `__graft_entry__.build()`.
The shared object is written next to the sources (`pytorch_fem_solver_b200/lib/`) so it
travels with the repository snapshot to the GPU box; nothing is JIT-compiled at import.
"""

from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB_DIR = os.path.join(PKG, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libtfem_b200.so")
STAMP = os.path.join(LIB_DIR, "libtfem_b200.stamp")
SOURCES = ["geometry.cu", "forms.cu", "scatter.cu", "interp.cu", "sparse.cu", "symbolic.cu", "topology.cu", "mlp.cu", "assemble_tiled.cu", "amg.cu"]
NVCC_FLAGS = [
    "-O3",
    "-std=c++17",
    "-gencode",
    "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-Xcompiler",
    "-fPIC",
    "-Xptxas=-v",
]


def _nvcc() -> str:
    for candidate in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if candidate and os.path.exists(candidate):
            return candidate
    raise RuntimeError("nvcc not found: the tfem_b200 CUDA library cannot be built")


def _digest() -> str:
    h = hashlib.sha256()
    paths = [os.path.join(CSRC, s) for s in SOURCES] + [
        os.path.join(CSRC, "common.cuh"),
        os.path.join(REPO, "include", "tfem_b200.h"),
    ]
    for path in paths:
        with open(path, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH) or not os.path.exists(STAMP):
        return True
    with open(STAMP) as fh:
        return fh.read().strip() != _digest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu for sm_100a and link libtfem_b200.so; returns its path."""
    if not force and not needs_build():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    nvcc = _nvcc()
    objects = []
    log = []
    for src in SOURCES:
        obj = os.path.join(LIB_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-I", os.path.join(REPO, "include"), "-I", CSRC, "-c", os.path.join(CSRC, src), "-o", obj]
        proc = subprocess.run(cmd, capture_output=True, text=True)
        log.append(proc.stderr)
        if proc.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{proc.stdout}\n{proc.stderr}")
        objects.append(obj)
    link = [nvcc, "-shared", "-o", LIB_PATH, *objects, "-cudart", "static"]
    proc = subprocess.run(link, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError(f"link failed:\n{proc.stdout}\n{proc.stderr}")
    with open(os.path.join(LIB_DIR, "ptxas.log"), "w") as fh:
        fh.write("\n".join(log))
    with open(STAMP, "w") as fh:
        fh.write(_digest())
    if verbose:
        print("\n".join(log))
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
