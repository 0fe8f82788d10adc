"""Build `pyslam_b200/libb2v.so` (the C-ABI library of include/b2v.h) in-tree with nvcc for sm_100a.

nvcc cross-compiles without a GPU; the resulting .so travels with the repo snapshot to the GPU
box.  `python -m pyslam_b200.build` or `pyslam_b200.build.build()`.
"""

from __future__ import annotations

import os
import shutil
import subprocess
import sys

_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_DIR, "csrc")
LIB = os.path.join(_DIR, "libb2v.so")
SOURCES = ["b2v_api.cu", "b2v_tsdf.cu", "b2v_mesh.cu", "b2v_grid.cu", "b2v_prep.cu", "b2v_semantic.cu"]
HEADERS = ["b2v_device.cuh", "b2v_internal.h", "b2v_points.cuh", "b2v_scan.cuh", "mc_tables.h", "../../include/b2v.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    # IEEE everywhere: no fast-math, no flush-to-zero, correctly rounded div/sqrt; FMA contraction is
    # left on for non-contract code only (contract code uses explicit-rounding intrinsics)
    "--ftz=false", "--prec-div=true", "--prec-sqrt=true",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-O2",
]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built")


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu for sm_100a and link libb2v.so.  Returns the library path."""
    if not force and not _stale():
        return LIB
    nvcc = _nvcc()
    env = dict(os.environ)
    # the image exports CC/CXX pointing at a wrapper; nvcc must use the system host compiler
    ccbin = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else (shutil.which("g++") or "g++")
    objdir = os.path.join(_DIR, "build")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, "-ccbin", ccbin, *NVCC_FLAGS, "-Xptxas", "-v", "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                                            text=True, env=env)))
        objs.append(obj)
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"==== {src} ====\n{out}")
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
    with open(os.path.join(objdir, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    cmd = [nvcc, "-ccbin", ccbin, "-shared", "-gencode", "arch=compute_100a,code=sm_100a",
           *objs, "-o", LIB]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
